"""Fixed-lambda fits on the whole C2 feature space (200 000 x 500 bp, k = 1..8 revcomp, matrix-free) with the
accelerated solver (FISTA with gradient restart, kmerlr_proxgrad_accel_full) and with fixed-step ISTA
(kmerlr_proxgrad), at the lambda of the first leapfrog selection for N = 10 and N = 100 (kmerlr_select at theta = 0).
FISTA runs to EpsilonLoss 1e-8; ISTA to the same stop under a fixed iteration budget.  Per fit: iterations, restarts,
device seconds, the objective F = f + lambda |theta_{1:}|_1 at the end and the nonzero count.  Then the cost of one
iteration of either solver from fixed-count runs (Epsilon = EpsilonLoss = 0), the two alternated: C2 matrix-free, C2
on the stored rows, and a binarized one-GPU C3 set (k = 1..10, 200 bp) at a stated fraction of its 2 M rows.  Prints the
card's name and power limit beside the numbers.
python tools/fixed_probe.py [out.json] [ista_budget] [c3_fraction]"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np

import kmerlr_b200 as K
from kmerlr_b200 import synth


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                                      text=True).strip()
        name, power = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power}
    except (OSError, subprocess.CalledProcessError, ValueError):
        return {"name": "unknown", "power_limit": "unknown"}


def first_lambda(d, N):
    s = K.featureSelector(np.ones(2), False, N, d.m, 0.0, K.TIE_INDEX)
    _, lam, ok = s.Select(d, 0.0, np.zeros(0, dtype=np.int64), np.zeros(0), 0.0)
    assert ok
    return float(lam)


def fit(d, lam, accelerated, eps_loss, max_iter):
    est = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=eps_loss, MaxIterations=max_iter, Accelerated=accelerated)
    est.Theta = np.zeros(d.m + 1)
    t0 = time.perf_counter()
    it, delta = est.estimate_proximal(d, lam)
    wall = time.perf_counter() - t0
    dev = K.last_device_ms() / 1e3
    obj = K.logisticRegression(est.Theta, est.ClassWeights, lam).Loss(d)
    r = {"iterations": int(it), "restarts": int(est.accel_state[3]) if accelerated else 0, "device_s": dev, "wall_s": wall,
         "objective": float(obj), "nonzero": int(np.count_nonzero(est.Theta[1:])),
         "converged": bool(it < max_iter), "max_iterations": int(max_iter)}
    print("  %s lambda %.6g: %7d iterations%s, %5d restarts, %8.3f s device, F %.12f, %d nonzero" % (
        "fista" if accelerated else "ista ", lam, it, "" if r["converged"] else " (budget, not converged)",
        r["restarts"], dev, obj, r["nonzero"]), flush=True)
    return r


def per_iteration(d, lam, iters, reps=3, label=""):
    """device ms per iteration of fixed-count runs, ISTA and FISTA alternated; the first round warms up both"""
    res = {False: [], True: []}
    for rep in range(reps + 1):
        for acc in (False, True):
            est = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=0.0, MaxIterations=iters, Accelerated=acc)
            est.Theta = np.zeros(d.m + 1)
            it, _ = est.estimate_proximal(d, lam)
            assert it == iters
            if rep > 0:
                res[acc].append(K.last_device_ms() / iters)
    out = {"iterations_per_run": iters, "ista_ms_per_iter": res[False], "fista_ms_per_iter": res[True]}
    print("per iteration, %s: ista %s ms, fista %s ms" % (label, " ".join("%.4f" % v for v in res[False]),
                                                          " ".join("%.4f" % v for v in res[True])), flush=True)
    return out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    ista_budget = int(sys.argv[2]) if len(sys.argv) > 2 else 20000
    c3_fraction = float(sys.argv[3]) if len(sys.argv) > 3 else 0.25
    info = card()
    print("card: %s, power limit %s" % (info["name"], info["power_limit"]), flush=True)
    K.init(0)
    buf, off, y = synth.training_set(100000, 100000, 500)
    d = K.compile_test_data(None, K.NewKmerCounter(1, 8, revcomp=True), None, None, True, False, (buf, off))
    d.SetLabels(y)
    del buf, off
    result = {"card": info, "c2": {"n": int(d.n), "m": int(d.m), "nnz": int(d.nnz), "k": "1..8 revcomp", "L": 500},
              "epsilon_loss": 1e-8, "ista_budget": ista_budget, "fits": []}
    for N in (10, 100):
        lam = first_lambda(d, N)
        print("N = %d: lambda %.9g" % (N, lam), flush=True)
        result["fits"].append({"N": N, "lambda": lam, "fista": fit(d, lam, True, 1e-8, 10 ** 7),
                               "ista": fit(d, lam, False, 1e-8, ista_budget)})
    lam = result["fits"][0]["lambda"]
    cost = {"c2_matrix_free": per_iteration(d, lam, 200, label="C2 matrix-free")}
    K.option("implicit", 0)
    try:
        cost["c2_stored_rows"] = per_iteration(d, lam, 100, label="C2 stored rows")
    finally:
        K.option("implicit", 1)
    d.free()
    n3 = int(1000000 * c3_fraction)
    buf, off, y = synth.training_set(n3, n3, 200)
    d3 = K.compile_test_data(None, K.NewKmerCounter(1, 10, revcomp=True), None, None, True, True, (buf, off))
    d3.SetLabels(y)
    del buf, off
    cost["c3_binarized"] = dict(per_iteration(d3, first_lambda(d3, 10), 50, label="C3 binarized x %.2f" % c3_fraction),
                                fraction_of_c3_rows=c3_fraction, n=int(d3.n), m=int(d3.m), nnz=int(d3.nnz))
    d3.free()
    result["per_iteration"] = cost
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
