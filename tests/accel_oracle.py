"""Accelerated proximal gradient (FISTA with gradient restart) restated on the CPU oracle's routines: the gradient,
the loss, the step size and the stopping rule are the ones the oracle's ISTA (ko_proxgrad) calls, so the two loops
differ only in the momentum lines.  The reference has no such solver; this is the definition kmerlr_proxgrad_accel is
checked against (include/kmerlr_b200.h states the same iteration).

One iteration, from theta, y and t (a fresh start is y = theta, t = 1):
    g = grad f(y);  theta' = y - s g, soft-thresholded at s lambda for j >= 1
    eval_stopping(theta, theta', epsilon): theta = theta', stop (y and t stay)
    (y - theta').(theta' - theta) > 0: restart, t' = 1, y' = theta'
    else t' = (1 + sqrt(1 + 4 t^2)) / 2, y' = theta' + ((t - 1) / t') (theta' - theta)
    hook: the delta-loss test on F(y') = f(y') + lambda |y'_{1:}|_1
"""
import math

import numpy as np

from oracle import oracle as O


def proxgrad_accel(rmat, labels, theta, y=None, t=1.0, cw=(1.0, 1.0), lam=0.0, l2=0.0, step_factor=1.0, epsilon=0.0,
                   epsilon_loss=1e-8, max_iter=100000, hook=None):
    """-> dict(theta, y, t, iters, restarts, delta).  hook = [loss_old, loss_new], updated in place."""
    th = np.array(theta, dtype=np.float64)
    y = th.copy() if y is None else np.array(y, dtype=np.float64)
    s = O.step_size(rmat, l2, step_factor)
    thr = s * lam
    hk = hook if hook is not None else [float("nan"), float("nan")]
    it, restarts, delta = 0, 0, 0.0
    with np.errstate(all="ignore"):
        for i in range(max_iter):
            g = O.gradient(rmat, labels, y, cw)
            tn = y - s * g
            a = np.fmax(np.abs(tn[1:]) - thr, 0.0)                 # fmax: C's, a NaN operand gives the other one
            tn[1:] = np.where(tn[1:] >= 0.0, a, -a)
            it = i + 1
            stop, delta = O._eval_stopping(th, tn, epsilon)
            if stop:
                th = tn
                break
            d = tn - th
            if float(np.dot(y - tn, d)) > 0.0:
                t, y = 1.0, tn.copy()
                restarts += 1
            else:
                t1 = (1.0 + math.sqrt(1.0 + 4.0 * (t * t))) / 2.0
                y = tn + ((t - 1.0) / t1) * d
                t = t1
            th = tn
            hk[0], hk[1] = hk[1], hk[0]                            # kmerLr_estimator_hook.go:46-99
            if epsilon_loss != 0.0:
                hk[1] = O.loss(rmat, labels, y, cw, lam)
                if abs(hk[0] - hk[1]) < epsilon_loss:
                    break
    return dict(theta=th, y=y, t=t, iters=it, restarts=restarts, delta=delta)


class EstimatorState:
    """what the estimator carries between leapfrog targets: active indices, theta, lambda, the hook state"""

    def __init__(self):
        self.active_idx = np.zeros(0, dtype=np.int64)
        self.active_theta = np.zeros(1)
        self.lam = 0.0
        self.hook = [float("nan"), float("nan")]


def estimate_loop(mat, labels, cw, N, est, tie=O.TIE_GO118, epsilon_lambda=0.0, l2=0.0, step_factor=1.0, epsilon=0.0,
                  epsilon_loss=1e-8, max_iter=100000, max_epochs=0):
    """ko_estimate_loop (kmerLr_estimator.go:209-255) with the accelerated solver; the momentum restarts at every epoch
    (y = theta of the new reduced matrix, t = 1).  -> dict(epochs, lambdas, iters, restarts, objective)"""
    out = dict(epochs=0, lambdas=[], iters=[], restarts=[], objective=[])
    have_r = False
    while max_epochs == 0 or out["epochs"] < max_epochs:
        r = O.select(mat, labels, cw, N, est.active_theta[0], est.active_idx, est.active_theta[1:], tie=tie,
                     epsilon_lambda=epsilon_lambda, prev_lambda=est.lam * mat.n)
        if not r["ok"] and have_r:
            break
        lam = r["lam"]
        est.lam = lam
        sel = np.nonzero(r["mask"])[0]
        th = np.zeros(len(sel))
        th[0] = est.active_theta[0]
        for j, v in zip(est.active_idx, est.active_theta[1:]):
            if v != 0.0:
                th[np.searchsorted(sel, j)] = v
        rm = O.reduce(mat, sel)
        res = proxgrad_accel(rm, labels, th, cw=cw, lam=lam, l2=l2, step_factor=step_factor, epsilon=epsilon,
                             epsilon_loss=epsilon_loss, max_iter=max_iter, hook=est.hook)
        est.active_idx = sel[1:].copy()
        est.active_theta = res["theta"]
        out["lambdas"].append(lam)
        out["iters"].append(res["iters"])
        out["restarts"].append(res["restarts"])
        out["objective"].append(O.loss(rm, labels, res["theta"], cw, lam))
        out["epochs"] += 1
        have_r = True
    return out
