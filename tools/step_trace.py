#!/usr/bin/env python
"""Where the time of one bench.py step goes: the C2 step of bench.py's step_resident (extract, SetLabels,
one-iteration estimate_proximal on the resident sequences, per-kernel events on as in bench.py's timed loop)
under torch.profiler with CUDA activities.  For each of the three timed calls it reports the device time the
library measured, the GPU kernel / memcpy / memset time, the GPU idle time between the call's first and last
GPU activity, the time before the first and after the last activity inside the call, and the launches.

    python tools/step_trace.py [--config c2] [--steps 3] [--warmup 3] [--out FILE] [--kernels]

The library runs in the same process and CUDA context as torch, so CUPTI sees its kernels and copies.  A GPU
activity belongs to the call whose host range contains its start (every call ends in a device synchronise).
"""
import argparse
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = {"c2": (100000, 100000, 500, 1, 8, False), "small": (2000, 2000, 500, 1, 8, False)}
CALLS = ("extract", "labels", "proxgrad")
GPU_CATS = {"kernel": "kernel", "gpu_memcpy": "memcpy", "gpu_memset": "memset"}


def busy_union(iv):
    """total length of the union of [a, b) intervals"""
    tot, end = 0.0, None
    for a, b in sorted(iv):
        if end is None or a > end:
            tot += b - a
            end = b
        elif b > end:
            tot += b - end
            end = b
    return tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", help="also write the summary to this file")
    ap.add_argument("--kernels", action="store_true", help="list every GPU activity of the last traced step")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile, record_function
    import kmerlr_b200 as K
    from kmerlr_b200 import api, synth

    n_fg, n_bg, L, M, N, binarize = CONFIGS[args.config]
    K.init(0)
    torch.cuda.init()
    buf, off, labels = synth.training_set(n_fg, n_bg, L)
    counter = K.NewKmerCounter(M, N, revcomp=True, binarize=binarize)
    seqs = K.Sequences((buf, off))
    cw = np.ones(2)

    def step(rec):
        out = {}
        for name in CALLS:
            l0 = K.launch_count()
            with rec("step_trace/" + name):
                if name == "extract":
                    data = api._extract(counter, seqs, None, None, False)
                elif name == "labels":
                    data.SetLabels(labels)
                else:
                    est = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=1e-300, MaxIterations=1)
                    est.Theta = np.zeros(data.m + 1)
                    est.ClassWeights = cw
                    est.estimate_proximal(data, 1e-3)
            out[name] = (K.last_device_ms(), K.launch_count() - l0)
        data.free()
        return out

    class _Null:
        def __init__(self, *a):
            pass

        def __enter__(self):
            return self

        def __exit__(self, *a):
            return False

    for _ in range(args.warmup):
        step(_Null)
    torch.cuda.synchronize()
    K.api.profile(True)                       # bench.py's timed loop runs with the per-kernel events on
    dev = []
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            dev.append(step(record_function))
        torch.cuda.synchronize()
    K.api.profile(False)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]

    ranges = sorted((e["ts"], e["ts"] + e["dur"], e["name"].split("/", 1)[1]) for e in events
                    if e.get("ph") == "X" and str(e.get("name", "")).startswith("step_trace/") and e.get("cat") != "gpu_user_annotation")
    gpu = sorted((e["ts"], e["ts"] + e.get("dur", 0), GPU_CATS[e["cat"]], e["name"]) for e in events
                 if e.get("ph") == "X" and e.get("cat") in GPU_CATS)
    per = {c: {"wall": [], "kernel": [], "memcpy": [], "memset": [], "idle": [], "before": [], "after": [],
               "kernels": [], "copies": []} for c in CALLS}
    last_step = {}
    for i, (a, b, name) in enumerate(ranges):
        acts = [g for g in gpu if a <= g[0] < b]
        p = per[name]
        p["wall"].append(b - a)
        for cat in ("kernel", "memcpy", "memset"):
            p[cat].append(sum(g[1] - g[0] for g in acts if g[2] == cat))
        p["kernels"].append(sum(1 for g in acts if g[2] == "kernel"))
        p["copies"].append(sum(1 for g in acts if g[2] != "kernel"))
        if acts:
            first, last = acts[0][0], max(g[1] for g in acts)
            p["idle"].append((last - first) - busy_union([(g[0], g[1]) for g in acts]))
            p["before"].append(first - a)
            p["after"].append(b - last)
        else:
            p["idle"].append(0.0); p["before"].append(b - a); p["after"].append(0.0)
        if i >= len(ranges) - len(CALLS):
            last_step[name] = [(g[0] - a, g[1] - g[0], g[2], g[3]) for g in acts]

    us = lambda v: float(np.median(v)) if v else 0.0
    lines = ["step trace: config %s, %d traced steps after %d warm-up steps, per-kernel events on (as bench.py's timed loop)"
             % (args.config, args.steps, args.warmup),
             "medians over the steps, microseconds; device = the library's own event timing of the call (what bench.py adds up)",
             "%-9s %9s %9s %9s %9s %9s %9s %9s %9s %8s %8s" % ("call", "device", "host", "kernels", "memcpy", "memset",
                                                             "gpu idle", "pre-gpu", "post-gpu", "kernels", "copies")]
    tot = {k: 0.0 for k in ("device", "wall", "kernel", "memcpy", "memset", "idle", "before", "after")}
    launches = 0
    for c in CALLS:
        p = per[c]
        d = 1e3 * float(np.median([s[c][0] for s in dev]))
        row = {"device": d, "wall": us(p["wall"]), "kernel": us(p["kernel"]), "memcpy": us(p["memcpy"]),
               "memset": us(p["memset"]), "idle": us(p["idle"]), "before": us(p["before"]), "after": us(p["after"])}
        for k in tot:
            tot[k] += row[k]
        nk = int(np.median(p["kernels"])) if p["kernels"] else 0
        launches += nk
        lines.append("%-9s %9.1f %9.1f %9.1f %9.1f %9.1f %9.1f %9.1f %9.1f %8d %8d" % (
            c, row["device"], row["wall"], row["kernel"], row["memcpy"], row["memset"], row["idle"], row["before"],
            row["after"], nk, int(np.median(p["copies"])) if p["copies"] else 0))
    lines.append("%-9s %9.1f %9.1f %9.1f %9.1f %9.1f %9.1f %9.1f %9.1f %8d" % (
        "step", tot["device"], tot["wall"], tot["kernel"], tot["memcpy"], tot["memset"], tot["idle"], tot["before"],
        tot["after"], launches))
    busy = tot["kernel"] + tot["memcpy"] + tot["memset"]
    lines.append("outside the GPU's busy time: %.1f us of %.1f us device time (%.0f %%)"
                 % (tot["device"] - busy, tot["device"], 100.0 * (tot["device"] - busy) / max(tot["device"], 1e-9)))
    lines.append("library launch counter per step: " + ", ".join("%s %d" % (c, int(np.median([s[c][1] for s in dev]))) for c in CALLS))
    if args.kernels:
        lines.append("")
        lines.append("GPU activities of the last traced step (start relative to the call's host range, duration, us):")
        for c in CALLS:
            lines.append("  %s" % c)
            for t, d, cat, name in last_step.get(c, []):
                lines.append("    %9.1f %8.1f  %-6s %s" % (t, d, cat, name[:90]))
    text = "\n".join(lines)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    seqs.free()


if __name__ == "__main__":
    main()
