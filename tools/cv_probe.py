"""Cross-validation folds as row subsets of one resident matrix (kmerlr_matrix_subset) against re-extracting every fold's
training rows, on one GPU.  Two shapes, 5 folds each (fold = i mod 5):
  C4: 20 000 x 500 bp, k = 1..6 revcomp (pair features in the run);  C2: 200 000 x 500 bp, k = 1..8 revcomp.
Per fold:
  * building the training subset, against re-extracting the training rows from host buffers as bench.py's c4 leg does
    (host gather of the rows + kmerlr_extract, unfrozen);
  * one full-space gradient (single features) on the training subset, matrix-free and over the stored rows, beside the
    same two passes on the whole data set (device ms, median of 5 after a warm-up call), and the matrix-free row kernel
    (imp_pass) alone per row, also on fold 0's training rows in a random order.
One untimed subset and re-extraction go first (the first calls grow the device memory arena).
Then the whole 5-fold run through crossvalidation with the accelerated solver (C4: pair features, N = 20, at most 12
epochs per fold as in the c4 leg; C2: N = 10, at most 2 epochs per fold).  Prints the card's name and power limit beside
the numbers.
python tools/cv_probe.py [out.json] [c2_rows]"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np

import kmerlr_b200 as K
from kmerlr_b200 import api, synth


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                                      text=True).strip()
        name, power = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power}
    except (OSError, subprocess.CalledProcessError, ValueError):
        return {"name": "unknown", "power_limit": "unknown"}


def grad_ms(d, implicit, reps=5):
    lr = K.logisticRegression(np.zeros(d.m + 1), (1.0, 1.0), 0.0)
    K.option("implicit", implicit)
    try:
        lr.Gradient(None, d)
        ms = []
        for _ in range(reps):
            lr.Gradient(None, d)
            ms.append(K.last_device_ms())
    finally:
        K.option("implicit", 1)
    return float(np.median(ms))


def imp_pass_ns_per_row(d, reps=10):
    """device time of the matrix-free row kernel alone (imp_pass, CUDA events around every launch) per row: the part of
    the gradient that scales with the rows, without the table builds, the fold and the tail"""
    lr = K.logisticRegression(np.zeros(d.m + 1), (1.0, 1.0), 0.0)
    lr.Gradient(None, d)
    api.profile(True)
    try:
        for _ in range(reps):
            lr.Gradient(None, d)
        prof = api.profile_dump()
    finally:
        api.profile(False)
    return 1e6 * sum(v[0] for k, v in prof.items() if k.startswith("(imp_pass")) / reps / d.n


def shape(name, n, N, run_kw, run_targets):
    buf, off, y = synth.training_set(n // 2, n - n // 2, 500)
    lens = np.diff(off)
    kc = K.NewKmerCounter(1, N, revcomp=True)
    d = K.compile_test_data(None, kc, None, None, True, False, (buf, off))
    d.SetLabels(y)
    fold = K.cv_groups(d.n, 5)
    whole = {"grad_matrix_free_ms": grad_ms(d, 1), "grad_stored_ms": grad_ms(d, 0), "imp_pass_ns_per_row": imp_pass_ns_per_row(d)}
    # one untimed subset and one untimed re-extraction first: the first calls grow the device memory arena
    w = np.nonzero(fold != 0)[0]
    d.subset(w).free()
    K.compile_test_data(None, kc, None, None, True, False,
                        (np.concatenate([buf[off[i]:off[i + 1]] for i in w]),
                         np.concatenate([[0], np.cumsum(lens[w])]).astype(np.int64))).free()
    folds = []
    for f in range(5):
        tr = np.nonzero(fold != f)[0]
        t0 = time.perf_counter()
        s = d.subset(tr)
        sub_wall, sub_dev = time.perf_counter() - t0, K.last_device_ms()
        t0 = time.perf_counter()
        o = np.concatenate([[0], np.cumsum(lens[tr])]).astype(np.int64)
        b = np.concatenate([buf[off[i]:off[i + 1]] for i in tr])
        t_take = time.perf_counter() - t0
        ext = K.compile_test_data(None, kc, None, None, True, False, (b, o))
        ext_wall, ext_dev = time.perf_counter() - t0, K.last_device_ms()
        ext.free()
        del b
        row = {"fold": f, "n_train": int(len(tr)), "subset_wall_ms": 1e3 * sub_wall, "subset_device_ms": sub_dev,
               "reextract_wall_ms": 1e3 * ext_wall, "reextract_host_gather_ms": 1e3 * t_take, "reextract_device_ms": ext_dev,
               "grad_matrix_free_ms": grad_ms(s, 1), "grad_stored_ms": grad_ms(s, 0), "imp_pass_ns_per_row": imp_pass_ns_per_row(s)}
        s.free()
        folds.append(row)
        print("%s fold %d: subset %.2f ms (device %.2f) | re-extraction %.1f ms (host gather %.1f, device %.2f) | gradient "
              "matrix-free %.3f ms, stored %.3f ms" % (name, f, row["subset_wall_ms"], sub_dev, row["reextract_wall_ms"],
                                                      row["reextract_host_gather_ms"], ext_dev, row["grad_matrix_free_ms"],
                                                      row["grad_stored_ms"]), flush=True)
    # the training rows of fold 0 in a random order: the matrix-free pass then reads the packed words out of row order
    s = d.subset(np.random.default_rng(1).permutation(np.nonzero(fold != 0)[0]))
    shuffled = {"grad_matrix_free_ms": grad_ms(s, 1), "imp_pass_ns_per_row": imp_pass_ns_per_row(s)}
    s.free()
    print("%s whole data set: gradient matrix-free %.3f ms (imp_pass %.3f ns per row), stored %.3f ms; fold 0 in a random "
          "row order: matrix-free %.3f ms (imp_pass %.3f ns per row); imp_pass per row on the folds: %s" % (
              name, whole["grad_matrix_free_ms"], whole["imp_pass_ns_per_row"], whole["grad_stored_ms"],
              shuffled["grad_matrix_free_ms"], shuffled["imp_pass_ns_per_row"],
              ", ".join("%.3f" % r["imp_pass_ns_per_row"] for r in folds)), flush=True)
    t0 = time.perf_counter()
    cv = K.crossvalidation(d, fold, lambda: K.KmerLrEstimator(EpsilonLoss=1e-8, MaxIterations=10 ** 7, tie=K.TIE_INDEX,
                                                              Accelerated=True, **run_kw), run_targets)
    run_s = time.perf_counter() - t0
    print("%s 5-fold run: %.2f s, held-out loss %s" % (name, run_s, [round(float(x[-1]), 6) for x in cv.Loss]), flush=True)
    d.free()
    return {"shape": "%s: %d x 500 bp, k = 1..%d revcomp, m = %d" % (name, n, N, d.m), "whole": whole, "folds": folds,
            "fold0_shuffled": shuffled,
            "cv_run": {"s": run_s, "targets": list(run_targets), "estimator": run_kw, "solver": "accelerated",
                       "held_out_loss": [[float(v) for v in x] for x in cv.Loss],
                       "active": [int(len(m[-1][0])) for m in cv.Models]}}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    c2_rows = int(sys.argv[2]) if len(sys.argv) > 2 else 200000
    K.init(0)
    res = {"card": card()}
    print("card: %s, power limit %s" % (res["card"]["name"], res["card"]["power_limit"]), flush=True)
    res["c4"] = shape("C4", 20000, 6, {"Cooccurrence": True, "MaxEpochs": 12}, [20])
    res["c2"] = shape("C2", c2_rows, 8, {"MaxEpochs": 2}, [10])
    if out_path:
        os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
        with open(out_path, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
