"""Fixed-lambda fits over the pair-feature space at C4: the 16 000 training rows of fold 0 (k = 1..6 revcomp, m = 2 772,
3 843 379 coefficients, u32 counts) at the lambda of the first Select over the pair space for N = 20.

- the cost of one iteration by kernel, from kmerlr_profile (CUDA events around every launch, a run of its own): the row
  pass on the sparse term list (iterates from theta = 0) and on the O(q^2) walk (every pair coefficient non-zero),
  scatter_w, pairs_gradient, the prox step, the term list (flags, scan, emit) and pass_tail
- ISTA (kmerlr_proxgrad_pairs) under an iteration cap against FISTA (kmerlr_proxgrad_pairs_accel) to EpsilonLoss 1e-8:
  iterations, restarts, device seconds, F = f + lambda |theta_{1:}|_1 over every coefficient, non-zero single and pair
  coefficients
- the card's name and power limit, read in the same run
python tools/pair_fixed_probe.py [out.json] [ista_cap] [fista_cap]"""
import json
import os
import subprocess
import sys

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


def c4_fold0():
    buf, off, y = synth.training_set(10000, 10000, 500)
    n = len(off) - 1
    tr = np.nonzero(np.arange(n) % 5 != 0)[0]
    lens = np.diff(off)
    o = np.concatenate([[0], np.cumsum(lens[tr])]).astype(np.int64)
    b = np.concatenate([buf[off[i]:off[i + 1]] for i in tr])
    d = K.compile_test_data(None, K.NewKmerCounter(1, 6, revcomp=True), None, None, True, False, (b, o))
    d.SetLabels(y[tr].astype(np.uint8))
    return d


def objective(d, theta, lam):
    return K.logisticRegression(theta, (1.0, 1.0), 0.0, Cooccurrence=True).Loss(d) + lam * float(np.sum(np.abs(theta[1:])))


def fit(d, lam, accelerated, eps_loss, cap, dim):
    est = K.KmerLrEstimator(Cooccurrence=True, Epsilon=0.0, EpsilonLoss=eps_loss, MaxIterations=cap,
                            Accelerated=accelerated)
    est.Theta = np.zeros(dim)
    it, _ = est.estimate_proximal(d, lam)
    dev = K.last_device_ms() / 1e3
    th = est.Theta
    r = {"iterations": int(it), "restarts": int(est.accel_state[3]) if accelerated else 0, "device_s": dev,
         "objective": objective(d, th, lam), "nonzero_single": int(np.count_nonzero(th[1:d.m + 1])),
         "nonzero_pair": int(np.count_nonzero(th[d.m + 1:])), "stopped_by_cap": bool(it >= cap), "cap": int(cap),
         "epsilon_loss": eps_loss}
    print("  %s: %6d iterations%s, %4d restarts, %8.3f s device, F %.12f, %d single + %d pair non-zero" % (
        "fista" if accelerated else "ista ", it, " (cap)" if r["stopped_by_cap"] else "", r["restarts"], dev,
        r["objective"], r["nonzero_single"], r["nonzero_pair"]), flush=True)
    return r


KERNELS = {"row pass": "rows_kernel", "scatter_w": "scatter_w", "pairs_gradient": "pairs_gradient",
           "prox": "prox_", "momentum": "accel_momentum", "term list": "pair_", "scan": "scan_", "pass_tail": "pass_tail"}


def split(d, theta, lam, iters, accelerated):
    """device ms per launch of every kernel of the iteration, over `iters` iterations from theta (profiled run)"""
    api.profile(1)
    try:
        if accelerated:
            est = K.KmerLrEstimator(Cooccurrence=True, EpsilonLoss=0.0, MaxIterations=iters, Accelerated=True)
        else:
            est = K.KmerLrEstimator(Cooccurrence=True, EpsilonLoss=0.0, MaxIterations=iters)
        est.Theta = theta.copy()
        it, _ = est.estimate_proximal(d, lam)
        assert it == iters
        out = {}
        for k, sub in KERNELS.items():
            ms, n = api.profile_read(sub)
            out[k] = {"ms_total": ms, "launches": n, "ms_per_launch": ms / n if n else None}
    finally:
        api.profile(0)
    return out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    ista_cap = int(sys.argv[2]) if len(sys.argv) > 2 else 300
    fista_cap = int(sys.argv[3]) if len(sys.argv) > 3 else 5000
    info = card()
    print("card: %s, power limit %s" % (info["name"], info["power_limit"]), flush=True)
    K.init(0)
    d = c4_fold0()
    dim = K.CoeffIndex(d.m).Dim()
    s = K.featureSelector(np.ones(2), True, 20, d.m, 0.0, K.TIE_INDEX)
    _, lam, ok = s.Select(d, 0.0, np.zeros(0, dtype=np.int64), np.zeros(0), 0.0)
    assert ok
    lam = float(lam)
    print("C4 fold 0: n %d, m %d, %d coefficients; lambda (N = 20) %.9g" % (d.n, d.m, dim, lam), flush=True)
    result = {"card": info, "c4_fold0": {"n": int(d.n), "m": int(d.m), "coefficients": int(dim), "nnz": int(d.nnz),
                                         "k": "1..6 revcomp", "L": 500}, "lambda_N20": lam}
    split(d, np.zeros(dim), lam, 2, False)                                  # warm-up: step size, column view, modules
    sparse = split(d, np.zeros(dim), lam, 20, False)
    dense_theta = np.full(dim, 1e-12)
    dense_theta[0] = 0.0
    walk = split(d, dense_theta, 0.0, 3, False)
    accel = split(d, np.zeros(dim), lam, 20, True)
    result["per_launch_ms"] = {"ista_from_zero_sparse_list": sparse, "ista_dense_theta_q2_walk": walk,
                               "fista_from_zero_sparse_list": accel}
    for name, sp in (("sparse list", sparse), ("O(q^2) walk", walk)):
        print("per launch, %s: %s" % (name, ", ".join("%s %.4f ms" % (k, v["ms_per_launch"]) for k, v in sp.items()
                                                      if v["ms_per_launch"] is not None)), flush=True)
    result["fits"] = {"ista": fit(d, lam, False, 1e-8, ista_cap, dim), "fista": fit(d, lam, True, 1e-8, fista_cap, dim)}
    d.free()
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
