"""Window-scoring rates of every model kind stage 3 accepts (W = 200, step = 10 over --mbp Mbp unless stated):

  1 bench      nucleotide k = 1..8 revcomp, 100 features, linear (the bench.py model)
  2 gapped     gapped k = 4..8 revcomp, 100 features, linear
  3 strands    complement + reverse, k = 1..8, 100 features, linear
  4 classes50k linear model over 50 000 classes, k = 1..9 revcomp
  5 binarized  binarized, 20 000 classes and 200 pair features, k = 1..8 revcomp (window hit tables)
  6 wide       k = 1..13 revcomp, 400 features, W = 20 000, step = 1 000 (prefix rows in global memory)

Sequences are resident in HBM; windows/s come from device time (kmerlr_last_device_ms).  Each workload also scores
a bounded sample of windows with the CPU oracle, for a GPU / CPU ratio.  The card's name and power limit are read
in the same run.  --lib loads another build of the library (to compare two builds in one run); a workload that
build refuses is reported as refused.  --dump DIR writes the scores of workload 1 as float64 .npy.

    python tools/score_probe.py [--mbp 96] [--reps 3] [--lib path/to/libkmerlr_b200.so] [--dump DIR] [--only 1,2]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001 -- the rates stand without it, the report says what is missing
        return "unknown (%s)" % e, "unknown"


def observed_model(K, O, sample, M, N, n_feat, pairs=0, seed=0, binarize=False, **flags):
    """a model over n_feat classes observed in `sample` (+ pairs): what a trained model looks like"""
    rng = np.random.default_rng(seed)
    ocfg = O.make_config(M, N, binarize=binarize, **flags)
    ref = O.extract(ocfg, [sample])
    k, code = ref.classes()
    if ref.m < n_feat:
        raise SystemExit("sample too short for %d classes (%d observed)" % (n_feat, ref.m))
    pick = np.sort(rng.choice(ref.m, size=n_feat, replace=False))
    feats = [(i, i) for i in range(n_feat)]
    for _ in range(pairs):
        a, b = sorted(rng.choice(n_feat, 2, replace=False))
        feats.append((int(a), int(b)))
    theta = rng.normal(scale=0.05, size=(1, len(feats) + 1))
    km = dict(counter=K.NewKmerCounter(M, N, binarize=binarize, **flags), class_k=k[pick], class_code=code[pick],
              features=feats, theta=theta, summary="")
    om = dict(km, cfg=ocfg)
    return km, om


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mbp", type=float, default=96.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--lib", default=None)
    ap.add_argument("--dump", default=None)
    ap.add_argument("--only", default="1,2,3,4,5,6")
    ap.add_argument("--oracle-windows", type=int, default=2000)
    args = ap.parse_args()
    from kmerlr_b200 import _lib
    if args.lib:
        _lib.SO_PATH = os.path.abspath(args.lib)
    import kmerlr_b200 as K
    from kmerlr_b200 import synth
    from oracle import oracle as O
    from bench import canonical_classes
    O.build()
    K.init(0)
    name, power = card()
    ncontig = 24
    clen = int(args.mbp * 1e6) // ncontig
    buf = synth.random_bases(clen * ncontig, 3)
    off = np.arange(ncontig + 1, dtype=np.int64) * clen
    sample = bytes(synth.random_bases(200_000, 17)).decode()
    only = {int(x) for x in args.only.split(",")}
    rng = np.random.default_rng(9)

    def bench_model():
        ck, cc = canonical_classes(100, 1, 8)
        theta = rng.normal(scale=0.05, size=(1, len(ck) + 1))
        km = dict(counter=K.NewKmerCounter(1, 8, revcomp=True), class_k=ck, class_code=cc,
                  features=[(i, i) for i in range(len(ck))], theta=theta, summary="")
        return km, dict(km, cfg=O.make_config(1, 8, revcomp=True))

    workloads = [
        (1, "bench: nucleotide k=1..8 revcomp, 100 features, linear", bench_model, 200, 10),
        (2, "gapped k=4..8 revcomp, 100 features, linear",
         lambda: observed_model(K, O, sample[:5000], 4, 8, 100, seed=2, revcomp=True, alphabet="gapped-nucleotide"),
         200, 10),
        (3, "complement+reverse k=1..8, 100 features, linear",
         lambda: observed_model(K, O, sample, 1, 8, 100, seed=3, complement=True, reverse=True), 200, 10),
        (4, "linear, 50000 classes, k=1..9 revcomp",
         lambda: observed_model(K, O, sample, 1, 9, 50_000, seed=4, revcomp=True), 200, 10),
        (5, "binarized, 20000 classes + 200 pairs, k=1..8 revcomp",
         lambda: observed_model(K, O, sample, 1, 8, 20_000, pairs=200, seed=5, revcomp=True, binarize=True), 200, 10),
        (6, "k=1..13 revcomp, 400 features, linear, W=20000 step=1000",
         lambda: observed_model(K, O, sample, 1, 13, 400, seed=6, revcomp=True), 20_000, 1_000),
    ]
    seqs = K.Sequences((buf, off))
    results = []
    for wid, what, make, W, step in workloads:
        if wid not in only:
            continue
        km, om = make()
        g = K.genomicKmerLr([km])
        windows = ncontig * ((clen - W + step - 1) // step)
        rec = {"workload": wid, "what": what, "W": W, "step": step, "genome_mbp": args.mbp, "windows": windows,
               "card": name, "power_limit": power, "lib": args.lib or "in-tree"}
        try:
            ms = []
            for i in range(args.reps + 1):
                g.predict_resident(seqs, W, step)
                if i > 0:
                    ms.append(K.last_device_ms())
        except K.KmerLrError as e:
            rec["refused"] = str(e)
            results.append(rec)
            print(json.dumps(rec), flush=True)
            continue
        t = float(np.median(ms)) * 1e-3
        rec.update(ms=[round(x, 3) for x in ms], windows_per_sec=windows / t)
        # CPU oracle on the first windows of contig 0 (all cores)
        nw = max(1, min(args.oracle_windows, (clen - W) // step))
        sub = bytes(buf[:(nw - 1) * step + W + 1]).decode()
        t0 = time.perf_counter()
        ref = O.score_windows([om], [sub], W, step, threads=os.cpu_count() or 1)
        tc = time.perf_counter() - t0
        rec.update(oracle_windows=nw, oracle_windows_per_sec=nw / tc, gpu_over_cpu=(windows / t) / (nw / tc),
                   oracle_cores=os.cpu_count())
        if args.dump and wid == 1:
            total = sum(O.window_slots(clen, W, step) for _ in range(ncontig))
            out = g.predict_resident(seqs, W, step, fetch=True, total_slots=total)
            os.makedirs(args.dump, exist_ok=True)
            np.save(os.path.join(args.dump, "workload1_scores.npy"), out[:total])
            first = out[:nw]
            rec["oracle_max_abs_diff"] = float(np.max(np.abs(first - ref[:nw])))
        results.append(rec)
        print(json.dumps(rec), flush=True)
    seqs.free()
    return results


if __name__ == "__main__":
    main()
