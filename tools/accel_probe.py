"""The C2 leapfrog path to 10 / 25 / 50 / 100 features (1 GPU, `|g| desc, index asc` ties, EpsilonLoss = 1e-8) once with
the fixed-step ISTA solver and once with the accelerated one (FISTA with gradient restart, KmerLrEstimator(Accelerated=
True)).  Per target: epochs, iterations, restarts, seconds, lambda and the objective F = f + lambda |theta_{1:}|_1 at the
end of each epoch; then the cost of one iteration of either solver at 100 features from fixed-count runs.  Prints the
card's name and power limit beside the numbers.
python tools/accel_probe.py [out.json] [n_per_class]"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np

import kmerlr_b200 as K
from kmerlr_b200 import synth

TARGETS = (10, 25, 50, 100)


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                                      text=True).strip()
        name, power = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power}
    except (OSError, subprocess.CalledProcessError, ValueError):
        return {"name": "unknown", "power_limit": "unknown"}


def path(d, accelerated):
    est = K.KmerLrEstimator(EpsilonLoss=1e-8, MaxIterations=10 ** 9, tie=K.TIE_INDEX, Accelerated=accelerated)
    epoch_log = []
    solve = est.estimate_proximal
    side = [0.0]                         # time spent on the objective below, taken out of the target's seconds

    def logged(reduced, lam):
        it, delta = solve(reduced, lam)
        t0 = time.perf_counter()
        obj = K.logisticRegression(est.Theta, est.ClassWeights, lam).Loss(reduced)
        epoch_log.append({"lambda": float(lam), "iterations": int(it), "objective": float(obj), "active": len(est.Theta) - 1,
                          "restarts": int(est.accel_state[3]) if accelerated else 0})
        side[0] += time.perf_counter() - t0
        return it, delta

    est.estimate_proximal = logged
    out = []
    for n_feat in TARGETS:
        first, side[0] = len(epoch_log), 0.0
        t0 = time.perf_counter()
        epochs = est.estimate_loop(d, n_feat)
        s = time.perf_counter() - t0 - side[0]
        ep = epoch_log[first:]
        assert len(ep) == epochs
        out.append({"features": n_feat, "epochs": int(epochs), "iterations": int(sum(e["iterations"] for e in ep)),
                    "restarts": int(sum(e["restarts"] for e in ep)), "s": s, "lambda": float(est.path[-1][0]),
                    "epoch_log": ep})
        print("%s N=%3d: %2d epochs, %8d iterations, %5d restarts, %8.3f s, lambda %.6g, F %.9f" % (
            "accel" if accelerated else "ista ", n_feat, epochs, out[-1]["iterations"], out[-1]["restarts"], s,
            out[-1]["lambda"], ep[-1]["objective"]), flush=True)
    return out, np.concatenate([[0], est.active_idx]), est.path[-1][0]


def per_iteration(d, sel, lam, iters=20000, reps=3):
    """device time of fixed-count runs (Epsilon = EpsilonLoss = 0) on the reduced matrix of the 100-feature model,
    the two solvers alternated"""
    rd = K.select_data(d, sel)
    rd.SetLabels(d.Labels)
    res = {False: [], True: []}
    for rep in range(reps + 1):
        for acc in (False, True):
            est = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=0.0, MaxIterations=iters, Accelerated=acc)
            est.Theta = np.zeros(len(sel))
            it, _ = est.estimate_proximal(rd, lam)
            assert it == iters
            if rep > 0:                      # rep 0 warms up both
                res[acc].append(1e3 * K.last_device_ms() / iters)
    out = {"reduced_rows": int(rd.n), "reduced_nnz": int(rd.nnz), "iterations_per_run": iters,
           "ista_us_per_iter": res[False], "accel_us_per_iter": res[True]}
    rd.free()
    print("per iteration at %d features (nnz %d): ista %s us, accel %s us" % (
        len(sel) - 1, out["reduced_nnz"], " ".join("%.2f" % v for v in res[False]),
        " ".join("%.2f" % v for v in res[True])), flush=True)
    return out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    n = int(sys.argv[2]) if len(sys.argv) > 2 else 100000
    info = card()
    print("card: %s, power limit %s" % (info["name"], info["power_limit"]), flush=True)
    K.init(0)
    buf, off, y = synth.training_set(n, n, 500)
    d = K.compile_test_data(None, K.NewKmerCounter(1, 8, revcomp=True), None, None, True, False, (buf, off))
    d.SetLabels(y)
    result = {"card": info, "data": {"n": int(d.n), "m": int(d.m), "nnz": int(d.nnz), "k": "1..8 revcomp", "L": 500},
              "epsilon_loss": 1e-8, "tie": "index"}
    for acc in (False, True):
        t0 = time.perf_counter()
        legs, sel, lam = path(d, acc)
        result["accel" if acc else "ista"] = {"targets": legs, "path_s": time.perf_counter() - t0}
    result["per_iteration_at_100"] = per_iteration(d, sel, lam)
    d.free()
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
