#!/usr/bin/env python
"""bench.py -- the kmerLr hot path on B200: k-mer sequences/sec (+ prox-grad iterations/sec).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU algorithm (oracle port)
    python bench.py ... --dump-outputs DIR                    # also write what the last timed step computed (.npy)

One STEP = one pass of the hot path over one batch of synthetic input of the BASELINE.json
configs[1] shape (C2): extract 100 000 fg + 100 000 bg sequences x 500 bp, k = 1..8, revcomp-merged,
into the sparse count matrix, then one full-space proximal-gradient iteration on it (one pass: z, loss,
weights, X^T w; prox update; then the hook's loss at the new theta).  N > 1: every rank (GPU) gets its own
200 000-sequence shard (weak scaling); the class union and the gradient are reduced over NCCL.
Beside the headline the line carries: full-space iterations/s, reduced-matrix (100 columns) iterations/s,
sliding-window scoring on a bounded genome, the roofline of the dominant kernel, clocks, the CPU baseline.

`value` is timed on the device (CUDA events on the library's stream) with the packed sequences
already resident in HBM; `e2e` is the same step through the host-buffer C-ABI calls
(kmerlr_extract + kmerlr_proxgrad) with the H2D / D2H copies inside a wall-clock region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (n_fg, n_bg, L, M, N, binarize)
    "c2": (100000, 100000, 500, 1, 8, False),
    "c3": (1000000, 1000000, 200, 1, 10, True),
    "small": (2000, 2000, 500, 1, 8, False),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, sm_load, mx, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
                if len(r) > 7 and float(r[7]) >= 10.0:       # the GPU was busy in this sample's window
                    sm_load.append(float(r[0]))
            except Exception:
                pass
        use = sm_load if sm_load else sm
        return {"sm_mhz": float(np.median(use)) if use else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "samples_under_load": len(sm_load), "reasons": sorted(reasons)}


def algorithmic_bytes_extract(n, L, nnz, binarize):
    """SURVEY 8d / BASELINE.md 4: ceil(L/4) + q (4 + v) + 8 per sequence"""
    return n * ((L + 3) // 4) + nnz * (4 + (0 if binarize else 4)) + n * 8


def algorithmic_bytes_iter(n, m, nnz, binarize):
    """nnz (4 + v) + (n+1) 8 + n + 3 (m+1) 8 per full-space prox-grad iteration"""
    return nnz * (4 + (0 if binarize else 4)) + (n + 1) * 8 + n + 3 * (m + 1) * 8


def dump_outputs(out_dir, data, est, sample_rows=1024, seed=0, budget=64 << 20):
    """what one step hands its caller, as out_dir/<name>.npy in float64: the estimator's theta and the hook's loss
    at that theta, the class list (k, code), the entry count of every row of the count matrix, and the entries of
    a fixed, seeded sample of its rows -- as many of the sampled rows as fit in `budget` bytes in all.  The hook's
    loss_old is left out: a step runs one iteration, so it is still the NaN that stands for "no previous loss"."""
    rowptr, col, val = data.rows()
    k, code = data.Kmers()
    out = {"theta": est.Theta, "loss": est.hook_state[1:], "kmers_k": k, "kmers_code": code, "row_nnz": np.diff(rowptr)}
    left = budget - sum(8 * len(v) for v in out.values()) - 9 * 128 - 8      # 9 .npy headers, the first row pointer
    pick = np.random.default_rng(seed).permutation(data.n)[:sample_rows]
    # a row costs its row index, its row pointer and 16 bytes per entry
    cost = np.cumsum(16 + 16 * (rowptr[pick + 1] - rowptr[pick]))
    pick = np.sort(pick[:int(np.searchsorted(cost, max(left, 0), side="right"))])
    ent = np.concatenate([np.arange(rowptr[r], rowptr[r + 1]) for r in pick]) if len(pick) else np.zeros(0, dtype=np.int64)
    out.update(sample_rows=pick, sample_rowptr=np.concatenate([[0], np.cumsum(rowptr[pick + 1] - rowptr[pick])]),
               sample_col=col[ent], sample_val=val[ent])
    out = {name: np.asarray(v, dtype=np.float64) for name, v in out.items()}
    bad = [name for name, v in out.items() if not np.all(np.isfinite(v))]
    if bad:
        raise ValueError("the last timed step computed non-finite values in: " + ", ".join(bad))
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)


def canonical_classes(n_classes, M, N, seed=5):
    """n_classes random revcomp classes (k, min(code, revcomp code)), sorted by (k, code)"""
    rng = np.random.default_rng(seed)
    out = set()
    while len(out) < n_classes:
        k = int(rng.integers(max(M, 4), N + 1))
        u = int(rng.integers(0, 4 ** k))
        r, x = 0, u
        for _ in range(k):
            r = (r << 2) | (3 - (x & 3))
            x >>= 2
        out.add((k, min(u, r)))
    cl = sorted(out)
    return np.array([c[0] for c in cl], dtype=np.int32), np.array([c[1] for c in cl], dtype=np.uint64)


def bench_scoring(K, mbp, rank, reps=3):
    """stage 3 (C5 shape at a bounded size): sliding-window scoring, W = 200, step = 10, of `mbp` Mbp in 24
    contigs with a 100-feature k = 1..8 revcomp count model; sequences resident in HBM, scores stay in HBM"""
    from kmerlr_b200 import synth
    W, step, ncontig = 200, 10, 24
    clen = int(mbp * 1e6) // ncontig
    buf = synth.random_bases(clen * ncontig, 3, offset=rank * clen * ncontig)
    off = np.arange(ncontig + 1, dtype=np.int64) * clen
    ck, cc = canonical_classes(100, 1, 8)
    rng = np.random.default_rng(9)
    theta = rng.normal(scale=0.05, size=(1, len(ck) + 1))
    model = dict(counter=K.NewKmerCounter(1, 8, revcomp=True), class_k=ck, class_code=cc,
                 features=[(i, i) for i in range(len(ck))], theta=theta, summary="")
    g = K.genomicKmerLr([model])
    seqs = K.Sequences((buf, off))
    windows = ncontig * ((clen - W + step - 1) // step)
    ms = []
    for i in range(reps + 1):
        g.predict_resident(seqs, W, step)
        if i > 0:
            ms.append(K.last_device_ms())
    seqs.free()
    t = float(np.mean(ms)) * 1e-3
    # the general kernel (binarized counts or pair features: a warp recounts every window) on a sixteenth of the slice
    glen = max(clen // 16, 4 * W)
    gmodel = dict(model, counter=K.NewKmerCounter(1, 8, revcomp=True, binarize=True),
                  features=[(i, i) for i in range(len(ck))] + [(0, 1), (2, 5), (3, 4)],
                  theta=rng.normal(scale=0.05, size=(1, len(ck) + 4)))
    gg = K.genomicKmerLr([gmodel])
    goff = np.arange(ncontig + 1, dtype=np.int64) * glen
    gseqs = K.Sequences((buf[:glen * ncontig], goff))
    gms = []
    for i in range(3):
        gg.predict_resident(gseqs, W, step)
        if i > 0:
            gms.append(K.last_device_ms())
    gseqs.free()
    gt = float(np.mean(gms)) * 1e-3
    gwin = ncontig * ((glen - W + step - 1) // step)
    generic = {"what": "score_generic: binarized model with 3 pair features, %d bp per contig" % glen, "ms": 1e3 * gt,
               "windows_per_sec": gwin / gt, "bases_per_sec": glen * ncontig / gt}
    return {"generic_kernel": generic,
            "windows_per_sec": windows / t, "bases_per_sec": clen * ncontig / t, "ms": 1e3 * t, "genome_mbp": mbp,
            "window": W, "step": step, "model_features": int(len(ck)), "algorithmic_bytes_per_window": step / 4 + 8,
            "achieved_gbs": windows * (step / 4 + 8) / t / 1e9,
            # the honest bound of this stage is integer throughput: one class-table probe per base and level
            "probes_per_sec": clen * ncontig * 8 / t, "probes_per_base": 8,
            "model": model, "sample": (buf, off)}



def leg_c3(K, api, synth, shard, rank, world, dist, allmax, allsum, peak, iters=10, reps=3):
    """BASELINE configs[2]: ONE set of 2 M sequences x 200 bp, k = 1..10 binarized, revcomp-merged, sample-sharded over
    the ranks (strong scaling): extraction of the rank's shard (class union OR-ed over NCCL), then full-space
    proximal-gradient iterations with the int64 all-reduce of the (m+1)-word fixed-point gradient"""
    import numpy as np
    n_fg, n_bg, L, M, N, binarize = CONFIGS["c3"]
    lo, hi = shard.sample_range(n_fg + n_bg, rank, world)
    f_lo, f_hi, b_lo, b_hi = min(lo, n_fg), min(hi, n_fg), max(lo - n_fg, 0), max(hi - n_fg, 0)
    fb, fo = synth.sequences(f_hi - f_lo, L, 1, planted=True, first=f_lo)
    bb, bo = synth.sequences(b_hi - b_lo, L, 2, planted=False, first=b_lo)
    buf = np.concatenate([fb, bb])
    off = np.concatenate([fo, bo[1:] + fo[-1]])
    labels = np.concatenate([np.ones(f_hi - f_lo, dtype=np.uint8), np.zeros(b_hi - b_lo, dtype=np.uint8)])
    counter = K.NewKmerCounter(M, N, revcomp=True, binarize=binarize)
    seqs = K.Sequences((buf, off))
    sharded = world > 1
    for opt in ("persist_bps", "p2p_allreduce", "super_len", "fused_ticket", "small_long"):       # experiments: KMERLR_OPT_<NAME>=value
        if os.environ.get("KMERLR_OPT_" + opt.upper()):
            K.option(opt, int(os.environ["KMERLR_OPT_" + opt.upper()]))
    ext = []
    data = None
    for i in range(reps + 1):
        if data is not None:
            data.free()
        data = api._extract(counter, seqs, None, None, sharded)
        if i > 0:
            ext.append(K.last_device_ms())
    data.SetLabels(labels)
    est = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=1e-300, MaxIterations=2)
    est.Theta = np.zeros(data.m + 1)
    est.estimate_proximal(data, 1e-3)
    est.MaxIterations = iters
    its = []
    for rep in range(4):                         # one more warm-up at this length (the arena settles), then 3 timed
        est.Theta = np.zeros(data.m + 1)
        if dist is not None:
            dist.barrier()
        est.estimate_proximal(data, 1e-3)
        if rep > 0:
            its.append(K.last_device_ms() / iters)
    it_ms = float(np.median(its))                # timed without the per-kernel events
    est.Theta = np.zeros(data.m + 1)
    K.api.profile(True)
    est.estimate_proximal(data, 1e-3)            # the same iterations again for the per-kernel split
    it_ms_prof = K.last_device_ms() / iters
    prof = K.api.profile_dump()
    K.api.profile(False)
    ar_ms = sum(v[0] for k, v in prof.items() if k.startswith("nccl_") or "p2p_allreduce" in k) / iters
    pass_ms = sum(v[0] for k, v in prof.items() if "imp_pass" in k or "fused_kernel" in k or "low_accumulate" in k) / iters
    other_ms = sum(v[0] for k, v in prof.items()) / iters - ar_ms - pass_ms
    n_loc, m, nnz_loc = data.n, data.m, data.nnz
    data.free(); seqs.free()
    ext_ms, it_ms, ar_ms, pass_ms = allmax(float(np.mean(ext))), allmax(it_ms), allmax(ar_ms), allmax(pass_ms)
    nnz = int(allsum(float(nnz_loc)))
    n = n_fg + n_bg
    it_bytes = algorithmic_bytes_iter(n, m, nnz, binarize)
    ex_bytes = algorithmic_bytes_extract(n, L, nnz, binarize)
    return {"workload": "C3: 2 000 000 sequences x 200 bp in total, k=1..10 binarized, revcomp-merged, contiguous sample "
                        "shards over %d GPU(s) (strong scaling)" % world,
            "n_total": n, "n_per_gpu": int(n_loc), "m": int(m), "nnz_total": nnz,
            "extract_ms": ext_ms, "extract_sequences_per_sec": n / (ext_ms * 1e-3),
            "extract_frac_of_hbm_peak": ex_bytes / world / (ext_ms * 1e-3) / 1e9 / peak,
            "ms_per_iter": it_ms, "iters_per_sec": 1e3 / it_ms, "logistic_pass_ms": pass_ms,
            "other_kernels_ms_per_iter": other_ms, "ms_per_iter_with_kernel_events": it_ms_prof,
            "allreduce_ms_per_iter": ar_ms, "allreduce_share_of_iter": ar_ms / it_ms if it_ms > 0 else None,
            "allreduce_bytes": 8 * (m + 1), "algorithmic_bytes_per_iter": it_bytes,
            "allreduce_path": ("NVLink peer memory (two-shot, one cooperative launch)" if os.environ.get("KMERLR_OPT_P2P_ALLREDUCE", "0") not in ("", "0") else "NCCL int64 sum") if world > 1 else None,
            "iter_achieved_gbs_per_gpu": it_bytes / world / (it_ms * 1e-3) / 1e9,
            "iter_frac_of_hbm_peak": it_bytes / world / (it_ms * 1e-3) / 1e9 / peak}


def leg_path(K, synth, targets=(10, 25, 50, 100)):
    """BASELINE configs[1] as it is worded: the proximal-gradient leapfrog path to 100 features on the C2 set
    (1 GPU; EpsilonLoss = 1e-8 as the CLI default, `|g| desc, index asc` tie rule).  The last target alone needs
    ~1.5 M iterations of the reference's fixed-step ISTA (minutes): the default bench stops at 50 features and
    `--legs path100` runs the whole path (profiles/r02_path_to_100.json holds that run)."""
    n_fg, n_bg, L, M, N, _ = CONFIGS["c2"]
    buf, off, y = synth.training_set(n_fg, n_bg, L)
    t0 = time.perf_counter()
    d = K.compile_test_data(None, K.NewKmerCounter(M, N, revcomp=True), None, None, True, False, (buf, off))
    d.SetLabels(y)
    t_extract = time.perf_counter() - t0
    est = K.KmerLrEstimator(EpsilonLoss=1e-8, MaxIterations=10 ** 9, tie=K.TIE_INDEX)
    out, t_all = [], time.perf_counter()
    for n_feat in targets:
        t0 = time.perf_counter()
        epochs = est.estimate_loop(d, n_feat)
        out.append({"features": n_feat, "epochs": int(epochs), "iterations": int(sum(p[1] for p in est.path[-epochs:])),
                    "lambda": float(est.path[-1][0]), "active": int(len(est.active_idx)), "s": time.perf_counter() - t0,
                    "reduced_nnz_last_epoch": int(est.path[-1][3])})
    total = time.perf_counter() - t_all
    d.free()
    return {("path_to_%d_features_s" % targets[-1]): total, "extract_s": t_extract, "iterations": int(sum(o["iterations"] for o in out)),
            "epochs": int(sum(o["epochs"] for o in out)), "targets": out,
            "note": "wall clock through the C ABI, estimate_loop per target warm-started as Estimate does "
                    "(kmerLr_estimator.go:257-270); iteration counts are those of the reference's fixed-step ISTA"}


def leg_c4(K, synth, n=20000, folds=5, n_feat=20, max_epochs=12, only=None):
    """BASELINE configs[3]: pair features over k = 1..6 (CoeffIndex.Dim = 3.84 M coefficients), leapfrog path to N = 20,
    5-fold cross-validation with fold = i mod 5 over fg||bg (no shuffle).  Per fold: extraction of the training rows,
    the pair gradient / Select of every epoch, the reduced solves, loss on the held-out fold."""
    import numpy as np
    buf, off, y = synth.training_set(n // 2, n // 2, 500)
    kc = K.NewKmerCounter(1, 6, revcomp=True)
    fold = np.arange(n) % folds
    out = []
    lens = np.diff(off)
    for f in range(folds):
        if only is not None and f not in only:           # several GPUs: the folds are independent replicas, rank r takes f = r mod N
            continue
        t_fold = time.perf_counter()
        tr, te = np.nonzero(fold != f)[0], np.nonzero(fold == f)[0]

        def take(rows):
            o = np.concatenate([[0], np.cumsum(lens[rows])]).astype(np.int64)
            b = np.concatenate([buf[off[i]:off[i + 1]] for i in rows]) if len(rows) else np.zeros(1, dtype=np.uint8)
            return b, o
        t0 = time.perf_counter()
        dtr = K.compile_test_data(None, kc, None, None, True, False, take(tr))
        dtr.SetLabels(y[tr])
        t_extract = time.perf_counter() - t0
        nt = K.CoeffIndex(dtr.m).Dim()
        lr = K.logisticRegression(np.zeros(nt), (1.0, 1.0), 0.0, Cooccurrence=True)
        lr.Gradient(None, dtr)                       # builds the transposed view once
        t0 = time.perf_counter()
        lr.Gradient(None, dtr)
        grad_wall, grad_dev = time.perf_counter() - t0, K.last_device_ms()
        sel = K.featureSelector((1.0, 1.0), True, n_feat, dtr.m, tie=K.TIE_INDEX)
        t0 = time.perf_counter()
        sel.Select(dtr, 0.0, [], [], 0.0)
        select_wall = time.perf_counter() - t0
        est = K.KmerLrEstimator(Cooccurrence=True, EpsilonLoss=1e-8, MaxIterations=10 ** 7, MaxEpochs=max_epochs, tie=K.TIE_INDEX)
        t0 = time.perf_counter()
        epochs = est.estimate_loop(dtr, n_feat)
        t_path = time.perf_counter() - t0
        # held-out loss with the fold's model (kmerLr_classifier.go:107-147 SelectData + Loss)
        feats = [K.CoeffIndex(dtr.m).Sub2Ind(int(i) - 1) for i in est.active_idx]
        dte = K.compile_test_data(None, kc, dtr.Kmers(), feats, False, False, take(te))
        dte.SetLabels(y[te])
        loss = K.logisticRegression(est.Theta, (1.0, 1.0), 0.0).Loss(dte)
        dtr.free(); dte.free()
        out.append({"fold": f, "n_train": int(len(tr)), "extract_s": t_extract, "pair_gradient_ms": grad_dev,
                    "pair_gradient_wall_ms": 1e3 * grad_wall, "select_wall_ms": 1e3 * select_wall, "epochs": int(epochs),
                    "iterations": int(sum(p[1] for p in est.path)), "path_s": t_path, "lambda": float(est.path[-1][0]),
                    "active": int(len(est.active_idx)), "test_loss": float(loss), "wall_s": time.perf_counter() - t_fold})
    return {"workload": "C4: %d sequences x 500 bp, k=1..6 revcomp, pair features (%d coefficients), N=%d, %d folds (fold = i mod %d)"
                        % (n, K.CoeffIndex(2772).Dim(), n_feat, folds, folds), "folds": out}


def c4_summary(c4, world):
    import numpy as np
    out = sorted(c4["folds"], key=lambda o: o["fold"])
    per_rank = {}
    for o in out:
        per_rank[o["fold"] % world] = per_rank.get(o["fold"] % world, 0.0) + o["wall_s"]
    c4.update({"folds": out, "pair_gradient_ms": float(np.mean([o["pair_gradient_ms"] for o in out])),
               "select_wall_ms": float(np.mean([o["select_wall_ms"] for o in out])),
               "fold_wall_s": float(np.mean([o["wall_s"] for o in out])),
               "cross_validation_wall_s": float(max(per_rank.values())),
               "replicas": "fold f on GPU f mod %d, no collective" % world if world > 1 else "one GPU, folds one after the other"})
    return c4


def leg_c5(K, lib, torch, rank, world, mbp=384.0):
    """BASELINE configs[4] at a bounded size per GPU: sliding-window scoring (W = 200, step = 10) through the
    host-buffer C-ABI call -- H2D of the ASCII contigs, packing, scoring, D2H of every window score inside the timer"""
    import ctypes as C
    import numpy as np
    from kmerlr_b200 import synth, _lib
    W, step, ncontig = 200, 10, 24
    clen = int(mbp * 1e6) // ncontig
    total = clen * ncontig
    pin = torch.empty(total, dtype=torch.uint8).pin_memory()
    pin.numpy()[:] = synth.random_bases(total, 3, offset=rank * total)
    off = np.arange(ncontig + 1, dtype=np.int64) * clen
    ck, cc = canonical_classes(100, 1, 8)
    theta = np.random.default_rng(9).normal(scale=0.05, size=(1, len(ck) + 1))
    model = dict(counter=K.NewKmerCounter(1, 8, revcomp=True), class_k=ck, class_code=cc,
                 features=[(i, i) for i in range(len(ck))], theta=theta, summary="")
    g = K.genomicKmerLr([model])
    slots = ncontig * int(lib.kmerlr_window_slots(clen, W, step))
    windows = ncontig * ((clen - W + step - 1) // step)
    out = torch.empty(slots, dtype=torch.float64).pin_memory()
    times = []
    for i in range(4):
        t0 = time.perf_counter()
        _lib.check(lib.kmerlr_score_windows(g._arr, 1, C.c_void_p(pin.data_ptr()), off.ctypes.data_as(C.c_void_p), ncontig,
                                            W, step, C.c_void_p(out.data_ptr())))
        if i > 0:
            times.append(time.perf_counter() - t0)
    t = float(np.mean(times))
    # the wiggle track of those scores (saveWindowPredictionsWiggle): records formatted on the device, host buffers on
    # both sides -- H2D of the scores (8 B per slot), D2H of the text (18 B per slot)
    text = torch.empty(18 * slots, dtype=torch.uint8).pin_memory()
    irr = C.c_int64(0)
    wt = []
    for i in range(3):
        t0 = time.perf_counter()
        _lib.check(lib.kmerlr_wiggle_records(C.c_void_p(out.data_ptr()), slots, C.c_void_p(text.data_ptr()), C.byref(irr)))
        if i > 0:
            wt.append(time.perf_counter() - t0)
    tw = float(np.mean(wt))
    wig = {"records": int(slots), "e2e_ms": 1e3 * tw, "e2e_records_per_sec": slots / tw, "text_bytes": int(18 * slots),
           "irregular_records": int(irr.value), "first_record": bytes(text.numpy()[:17]).decode()}
    return {"wiggle": wig, "workload": "C5 slice: %.0f Mbp per GPU in %d contigs, W=%d, step=%d, 100-feature k=1..8 model" % (mbp, ncontig, W, step),
            "e2e_windows_per_sec": windows / t, "e2e_bases_per_sec": total / t, "e2e_ms": 1e3 * t, "windows": int(windows),
            "h2d_bytes": int(total + off.nbytes), "d2h_bytes": int(8 * slots), "device_ms_last_call": K.last_device_ms(),
            "checksum": float(out.numpy()[:1000].sum())}


def run_reference(args, rank, world):
    """the reference's own CPU algorithm (oracle port: per-sequence hash-map counting, union + sort,
    O(n m) convert_counts walk, serial-over-samples gradient / loss) on the box's host cores"""
    if rank != 0:
        return
    from oracle import oracle as O
    from kmerlr_b200 import synth
    n_fg, n_bg, L, M, N, binarize = CONFIGS[args.config]
    cores = os.cpu_count() or 1
    s_fg = s_bg = max(1, min(n_fg, args.ref_sample // 2))
    cfg = O.make_config(M, N, revcomp=True, binarize=binarize)
    times = []
    for it in range(args.warmup + args.steps):
        buf, off, labels = synth.training_set(s_fg, s_bg, L, first_fg=it * s_fg, first_bg=it * s_bg)
        t0 = time.perf_counter()
        mat = O.extract(cfg, (buf, off), threads=cores, faithful=True)
        theta = np.zeros(mat.m + 1)
        O.proxgrad(mat, labels, theta, (1.0, 1.0), lam=1e-3, epsilon=0.0, epsilon_loss=1e-300, max_iter=1)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = (s_fg + s_bg) / (ms / 1e3)
    sample = "%d fg + %d bg sequences x %d bp per step (of %d + %d), k=%d..%d revcomp" % (s_fg, s_bg, L, n_fg, n_bg, M, N)
    line = {
        "impl": "reference", "metric": "kmer_sequences_per_sec", "value": value, "unit": "sequences/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": "sequences/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    n_fg, n_bg, L, M, N, binarize = CONFIGS[args.config]
    return {"workload": "%s: %d fg + %d bg sequences x %d bp per GPU, k=%d..%d, revcomp-merged%s; step = k-mer "
                        "extraction + one full-space proximal-gradient iteration" %
                        (args.config.upper(), n_fg, n_bg, L, M, N, ", binarized" if binarize else ""),
            "sequences_per_gpu": n_fg + n_bg, "seq_len": L, "k_min": M, "k_max": N,
            "parallelism": "sample-sharded x%d" % world,
            "l2": "working set larger than L2: every step writes the matrix rows (3.5 GB at C2) and re-reads the packed "
                  "sequences after them, so nothing survives in the 126 MB L2 from one step to the next"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--ref-sample", type=int, default=8000, help="sequences per step of the CPU arm")
    ap.add_argument("--iters", type=int, default=20, help="full-space prox-grad iterations timed back to back")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--score-mbp", type=float, default=96.0, help="genome size of the window-scoring leg (0 = skip)")
    ap.add_argument("--short", action="store_true", help="profiling runs only: allow fewer than 3 warm-up steps")
    ap.add_argument("--legs", default="auto", help="extra legs on the same JSON line: comma list of c3,path,path100,c4,c5; "
                    "auto = all four on one GPU, c3,c5 on several; none = headline only")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl ours")
    if args.warmup < 3 and args.impl == "ours" and not args.short:
        args.warmup = 3

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import kmerlr_b200 as K
    from kmerlr_b200 import api, synth

    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    K.init(local_rank)
    if world > 1:
        from kmerlr_b200 import shard
        cpus = shard.bind_host_to_gpu(local_rank)      # host buffers on the GPU's own socket
        if os.environ.get("KMERLR_BENCH_VERBOSE"):
            print("rank %d: %s host cpus local to the gpu" % (rank, len(cpus) if cpus else "no"), file=sys.stderr)
        K.comm_init_torch()
    sharded = world > 1

    n_fg, n_bg, L, M, N, binarize = CONFIGS[args.config]
    n = n_fg + n_bg
    buf, off, labels = synth.training_set(n_fg, n_bg, L, first_fg=rank * n_fg, first_bg=rank * n_bg)
    # pinned host copies (the e2e arm copies from pinned memory)
    pin = torch.empty(len(buf), dtype=torch.uint8).pin_memory()
    pin.numpy()[:] = buf
    hbuf = pin.numpy()
    counter = K.NewKmerCounter(M, N, revcomp=True, binarize=binarize)
    seqs = K.Sequences((hbuf, off))
    lam = 1e-3
    cw = np.ones(2)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident(keep=False):
        """returns (device ms, matrix info, (matrix, estimator) if keep else None: the caller frees that matrix)"""
        ms = 0.0
        data = api._extract(counter, seqs, None, None, sharded)
        ms += K.last_device_ms()
        data.SetLabels(labels)
        ms += K.last_device_ms()
        est = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=1e-300, MaxIterations=1)
        est.Theta = np.zeros(data.m + 1)
        est.ClassWeights = cw
        est.estimate_proximal(data, lam)
        ms += K.last_device_ms()
        info = (data.n, data.m, data.nnz)
        if keep:
            return ms, info, (data, est)
        data.free()
        return ms, info, None

    def step_e2e():
        """the same step through the host-buffer C-ABI calls; returns wall seconds"""
        t0 = time.perf_counter()
        data = api._extract(counter, (hbuf, off), None, None, sharded)
        data.SetLabels(labels)
        est = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=1e-300, MaxIterations=1)
        est.Theta = np.zeros(data.m + 1)
        est.ClassWeights = cw
        est.estimate_proximal(data, lam)
        checksum = float(est.Theta[0])          # the step's result, read on the host
        dt = time.perf_counter() - t0
        m = data.m
        data.free()
        return dt, m, checksum

    # clocks / throttle reasons are sampled every 20 ms from here to the end of the e2e loop: the warm-up
    # gives nvidia-smi time to start, every later phase is a timed region of one of the reported numbers
    sampler = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(args.warmup):
        step_resident()
    barrier()
    if sampler:
        sampler.rows.clear()             # keep only what is sampled from the first timed step on
    K.api.profile(True)
    launches0 = K.launch_count()
    dev_ms, info = [], None
    t_wall0 = time.perf_counter()
    for i in range(args.steps):
        ms, info, last = step_resident(keep=args.dump_outputs is not None and i == args.steps - 1)
        dev_ms.append(ms)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = K.launch_count() - launches0
    prof = K.api.profile_dump()
    K.api.profile(False)
    if last is not None:
        if rank == 0:
            dump_outputs(args.dump_outputs, *last)
        last[0].free()

    # full-space prox-grad iterations back to back on a resident matrix
    data = api._extract(counter, seqs, None, None, sharded)
    data.SetLabels(labels)
    est = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=1e-300, MaxIterations=2)
    est.Theta = np.zeros(data.m + 1)
    est.ClassWeights = cw
    est.estimate_proximal(data, lam)             # builds the CSC view, warms up
    est.MaxIterations = args.iters
    its = []
    for rep in range(4):                         # one more warm-up at this length (the arena settles), then 3 timed
        barrier()
        est.Theta = np.zeros(data.m + 1)
        est.estimate_proximal(data, lam)
        if rep > 0:
            its.append(K.last_device_ms())
    iter_ms = float(np.median(its))              # timed without the per-kernel events
    K.api.profile(True)
    est.Theta = np.zeros(data.m + 1)
    est.estimate_proximal(data, lam)             # the same iterations again for the per-kernel split
    prof_it = K.api.profile_dump()
    K.api.profile(False)
    n_rows, m_cols, nnz = data.n, data.m, data.nnz
    # iterations on a reduced matrix (100 columns, what the leapfrog path solves between selections)
    sel = np.unique(np.concatenate([[0], np.linspace(1, data.m, 100).astype(np.int64)]))
    rd = K.select_data(data, sel)
    rd.SetLabels(labels)
    red_iters = 2000
    try:
        est = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=0.0, MaxIterations=50)
        est.Theta = np.zeros(len(sel)); est.ClassWeights = cw
        lam_red = 1e-6                     # small enough that theta leaves 0 and the iterations keep running
        est.estimate_proximal(rd, lam_red)
        est.MaxIterations = red_iters
        est.Theta = np.zeros(len(sel))
        barrier()
        done_iters, _ = est.estimate_proximal(rd, lam_red)
        red_ms = K.last_device_ms()
        reduced = {"columns": int(len(sel) - 1), "nnz": int(rd.nnz), "iterations": int(done_iters),
                   "ms_per_iter": red_ms / max(done_iters, 1), "iters_per_sec": 1e3 * max(done_iters, 1) / red_ms,
                   "exchange": ("peer memory (NVLink mailboxes)" if os.environ.get("KMERLR_P2P", "1") != "0" else "NCCL") if world > 1 else None}
    except K.KmerLrError as e:           # a failed peer exchange must not take the headline numbers down
        reduced = {"error": str(e)}
        print("bench.py: reduced-matrix leg FAILED on rank %d: %s" % (rank, e), file=sys.stderr, flush=True)
    rd.free()
    data.free()

    # stage 3: sliding-window scoring on a bounded genome
    genomic = bench_scoring(K, args.score_mbp, rank) if args.score_mbp > 0 else None

    # e2e through host buffers
    e2e_s = []
    for i in range(2 + args.steps):                  # 2 untimed (the arena settles), then the timed ones
        dt, m_e2e, _ = step_e2e()
        if i > 1:
            e2e_s.append(dt)
    barrier()
    clocks = sampler.stop() if sampler else None

    def allmax(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    legs = args.legs
    if legs == "auto":
        legs = ("c3,path,c4,c5" if world == 1 else "c3,c4,c5") if args.config == "c2" else "none"
    legs = [x for x in legs.split(",") if x and x != "none"]
    seqs.free()
    extra = {}
    peak0, _ = peaks()
    from kmerlr_b200 import shard as shard_mod
    if "c3" in legs:
        extra["c3"] = leg_c3(K, api, synth, shard_mod, rank, world, dist, allmax, allsum, peak0)
    if "c5" in legs:
        c5 = leg_c5(K, K.api.lib(), torch, rank, world)
        ms5 = allmax(c5["e2e_ms"])
        c5["e2e_windows_per_sec"] = world * c5["windows"] / (ms5 * 1e-3)     # every rank its own contigs, no collective
        c5["e2e_bases_per_sec"] *= world * c5["e2e_ms"] / ms5
        c5["e2e_ms"] = ms5
        extra["c5"] = c5
    if rank == 0 and "path100" in legs:
        extra["c2_path"] = leg_path(K, synth)
    elif rank == 0 and "path" in legs:
        extra["c2_path"] = leg_path(K, synth, targets=(10, 25, 50))
        extra["c2_path"]["path_to_100_features_s"] = None
        try:
            extra["c2_path"]["path_to_100_features_measured_separately"] = json.load(open(os.path.join(ROOT, "profiles", "r02_path_to_100.json")))
        except Exception:
            pass
    if "c4" in legs:
        # the folds of a cross-validation are independent (kmerLr_crossvalidation.go:167-211): replicas over the GPUs
        c4 = leg_c4(K, synth, only=[f for f in range(5) if f % world == rank])
        if dist is not None:
            parts = [None] * world
            dist.all_gather_object(parts, c4["folds"])
            c4["folds"] = [o for p in parts for o in p]
        if rank == 0:
            extra["c4"] = c4_summary(c4, world)
    barrier()

    ms_step = allmax(float(np.mean(dev_ms)))
    ms_e2e = allmax(1e3 * float(np.mean(e2e_s)))
    ms_iter = allmax(iter_ms / args.iters)
    wall_ms_step = allmax(1e3 * t_wall / args.steps)
    if genomic is not None:
        gms = allmax(genomic["ms"])                  # slowest rank
        for key in ("windows_per_sec", "bases_per_sec", "achieved_gbs"):
            genomic[key] *= genomic["ms"] / gms
        genomic["ms"] = gms
    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    peak, peak_src = peaks()
    # dominant kernel of the step
    per_kernel = {k: v[0] / args.steps for k, v in prof.items()}
    merged = {}
    for k, v in per_kernel.items():
        nm = k.split("<")[0].strip("()")
        merged[nm] = round(merged.get(nm, 0.0) + v, 4)
    top = max(per_kernel, key=per_kernel.get)
    top_ms_total, top_launches = prof[top]
    if "extract_kernel" in top:
        abytes = algorithmic_bytes_extract(n_rows, L, nnz, binarize)
        what = "extraction: ceil(L/4) + q(4+v) + 8 bytes per sequence x %d sequences per launch" % n_rows
    else:
        abytes = algorithmic_bytes_iter(n_rows, m_cols, nnz, binarize)
        what = "one prox-grad pass"
    ach = abytes / (top_ms_total / top_launches * 1e-3) / 1e9
    ext_ms = sum(v for k, v in per_kernel.items() if "extract_kernel" in k)
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if args.config == "c2":
            traffic = tj.get(top.split("<")[0].strip("()"), {}).get("bytes")
    except Exception:
        pass
    roof = {"bound": "hbm", "kernel": top.split("<")[0].strip("()"), "achieved": ach, "peak": peak, "unit": "GB/s",
            "frac": ach / peak, "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": abytes,
            "what": what, "kernel_ms_per_launch": top_ms_total / top_launches,
            "kernel_share_of_step": per_kernel[top] / sum(per_kernel.values())}
    it_bytes = algorithmic_bytes_iter(n_rows, m_cols, nnz, binarize)
    it_fused = sum(v[0] for k, v in prof_it.items() if "fused_" in k) / max(1, sum(v[1] for k, v in prof_it.items() if "fused_" in k))
    line = {
        "metric": "kmer_sequences_per_sec", "value": world * n / (ms_step * 1e-3), "unit": "sequences/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world),
        "matrix": {"n": n_rows, "m": m_cols, "nnz": nnz},
        "e2e": {"value": world * n / (ms_e2e * 1e-3), "unit": "sequences/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(len(hbuf) + off.nbytes + labels.nbytes + 8 * (m_e2e + 1) + 64),
                "d2h_bytes_per_step": int(8 * (m_e2e + 1) + 64)},
        "gpu_launches": int(launches),
        "ms_steps": [round(x, 3) for x in dev_ms],
        "wall_ms_per_step": wall_ms_step,
        "extract_sequences_per_sec": world * n / (ext_ms * 1e-3) if ext_ms > 0 else None,
        "proxgrad_iters_per_sec": 1e3 / ms_iter,
        "proxgrad": {"ms_per_iter": ms_iter, "fused_pass_ms": it_fused,
                     "algorithmic_bytes_per_iter": it_bytes, "achieved_gbs": it_bytes / (ms_iter * 1e-3) / 1e9,
                     "frac_of_hbm_peak": it_bytes / (ms_iter * 1e-3) / 1e9 / peak},
        "reduced_proxgrad": reduced,
        "kernels_ms_per_step": dict(sorted(merged.items(), key=lambda kv: -kv[1])[:14]),
        "roofline": roof,
        "clocks": clocks,
    }
    line.update(extra)
    if genomic is not None:
        gmodel, gsample = genomic.pop("model"), genomic.pop("sample")
        if world > 1:
            genomic["windows_per_sec"] *= world       # every rank scores its own contigs, no collective
            genomic["bases_per_sec"] *= world
            genomic["achieved_gbs"] *= world
        genomic["frac_of_hbm_peak"] = genomic["achieved_gbs"] / world / peak
        line["genomic_scoring"] = genomic
    if world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as O
        cores = os.cpu_count() or 1
        if genomic is not None:
            # the reference's per-window recount on a bounded slice of the same genome
            nb = 400000
            omd = dict(cfg=O.make_config(1, 8, revcomp=True), class_k=gmodel["class_k"], class_code=gmodel["class_code"],
                       features=gmodel["features"], theta=gmodel["theta"], summary="")
            t0 = time.perf_counter()
            O.score_windows([omd], (gsample[0][:nb], np.array([0, nb], dtype=np.int64)), 200, 10, threads=cores)
            dtc = time.perf_counter() - t0
            genomic["cpu_baseline"] = {"windows_per_sec": ((nb - 200 + 9) // 10) / dtc, "cores": cores, "kind": "port",
                                       "sample": "%d bp of the same genome, all host threads" % nb}
        # the other legs: the same oracle port on a bounded sample of each leg's own shape (seconds each)
        if "c3" in extra:
            s3 = 3000
            b3, o3, l3 = synth.training_set(s3, s3, 200)
            t0 = time.perf_counter()
            m3 = O.extract(O.make_config(1, 10, revcomp=True, binarize=True), (b3, o3), threads=cores, faithful=True)
            t_e = time.perf_counter() - t0
            t0 = time.perf_counter()
            O.proxgrad(m3, l3, np.zeros(m3.m + 1), (1.0, 1.0), lam=lam, epsilon=0.0, epsilon_loss=1e-300, max_iter=1)
            t_i = time.perf_counter() - t0
            extra["c3"]["cpu_baseline"] = {"extract_sequences_per_sec": 2 * s3 / t_e, "iteration_rows_per_sec": 2 * s3 / t_i,
                                           "cores": cores, "kind": "port",
                                           "sample": "%d + %d sequences x 200 bp, k=1..10 binarized: extraction on all host threads, one "
                                                     "prox-grad iteration (serial over the samples, as the reference's Gradient is)" % (s3, s3)}
            extra["c3"]["iteration_rows_per_sec"] = extra["c3"]["n_total"] * extra["c3"]["iters_per_sec"]
        if "c4" in extra:
            s4 = 150
            b4, o4, l4 = synth.training_set(s4, s4, 500)
            m4 = O.extract(O.make_config(1, 6, revcomp=True), (b4, o4), threads=cores)
            t0 = time.perf_counter()
            O.gradient(m4, l4, np.zeros(O.ntheta(m4, True)), (1.0, 1.0), 0.0, cooccurrence=True)
            t_g = time.perf_counter() - t0
            extra["c4"]["cpu_baseline"] = {"pair_gradient_rows_per_sec": 2 * s4 / t_g, "cores": 1, "kind": "port",
                                           "sample": "%d + %d sequences x 500 bp, k=1..6 revcomp, every pair product of every row "
                                                     "(kmerLr_logistic_regression.go:200-216), serial over the samples" % (s4, s4)}
            extra["c4"]["pair_gradient_rows_per_sec"] = 16000 / (extra["c4"]["pair_gradient_ms"] * 1e-3)
        if "c5" in extra and "wiggle" in extra["c5"]:
            rng = np.random.default_rng(4)
            vals = -rng.random(20000) * 5
            t0 = time.perf_counter()
            for v in vals:
                O.go_fmt("%0.15f", O.go_exp(float(v)))
            extra["c5"]["wiggle"]["cpu_baseline"] = {"records_per_sec": len(vals) / (time.perf_counter() - t0), "cores": 1,
                                                     "kind": "port", "sample": "20 000 records through the Python restatement of "
                                                     "math.Exp + Fprintf (not Go's speed: a reference point for the checker only)"}
        s_half = max(1, min(n_fg, args.ref_sample // 2))
        sb, so, sl = synth.training_set(s_half, s_half, L)
        t0 = time.perf_counter()
        reps = 0
        while reps < 2 or time.perf_counter() - t0 < 10.0:
            mat = O.extract(O.make_config(M, N, revcomp=True, binarize=binarize), (sb, so), threads=cores, faithful=True)
            O.proxgrad(mat, sl, np.zeros(mat.m + 1), (1.0, 1.0), lam=lam, epsilon=0.0, epsilon_loss=1e-300, max_iter=1)
            reps += 1
            if time.perf_counter() - t0 > 30.0:
                break
        dt = (time.perf_counter() - t0) / reps
        line["cpu_baseline"] = {"value": 2 * s_half / dt, "unit": "sequences/s", "cores": cores, "kind": "port",
                                "sample": "%d fg + %d bg sequences x %d bp (of %d + %d), %d repetitions, all host "
                                          "threads; Go is not installed, so this is the C oracle port" %
                                          (s_half, s_half, L, n_fg, n_bg, reps)}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
