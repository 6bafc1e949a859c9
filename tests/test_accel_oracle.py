"""The accelerated proximal-gradient restatement (tests/accel_oracle.py) on the CPU: it reaches the optimum of TestScores1
that the ISTA oracle needs millions of iterations for, and it stops at a lower objective than ISTA under the same
delta-loss rule.  No GPU needed."""
import numpy as np
import pytest

import accel_oracle as A


@pytest.fixture(scope="module")
def scores1(oracle, fixtures):
    O = oracle
    X = np.vstack([fixtures["scoresLr_test_fg"], fixtures["scoresLr_test_bg"]])
    y = np.array([1] * 8 + [0] * 8, dtype=np.uint8)
    m = O.from_dense(X)
    r = O.select(m, y, (1, 1), 2, 0.0, [], [], tie=O.TIE_GO118)
    assert np.nonzero(r["mask"])[0].tolist() == [0, 2, 7]
    return O.reduce(m, [0, 2, 7]), y, r["lam"]


def test_scores1_reaches_the_optimum_in_hundreds_of_iterations(oracle, scores1):
    """SURVEY 0 finding 3: theta* = [0.851127, -0.054901, -0.030540] for features {1, 6} at lambda = 2.496875"""
    rm, y, lam = scores1
    assert "%e" % lam == "2.496875e+00"
    res = A.proxgrad_accel(rm, y, np.zeros(3), lam=lam, epsilon_loss=1e-13)
    assert 400 <= res["iters"] <= 1200, res["iters"]
    assert np.max(np.abs(res["theta"] - [0.851128, -0.054901, -0.030540])) <= 2e-6, res["theta"]
    assert res["restarts"] >= 1


def test_scores1_stops_below_ista_objective(oracle, scores1):
    """under EpsilonLoss = 1e-8 ISTA's delta-loss stop ends far from the optimum; the accelerated iterate ends lower"""
    O = oracle
    rm, y, lam = scores1
    res = A.proxgrad_accel(rm, y, np.zeros(3), lam=lam, epsilon_loss=1e-8)
    th, it, _ = O.proxgrad(rm, y, np.zeros(3), lam=lam, epsilon_loss=1e-8, max_iter=3000000)
    assert res["iters"] < it / 20
    assert O.loss(rm, y, res["theta"], lam=lam) < O.loss(rm, y, th, lam=lam)


def test_fresh_start_first_step_is_ista(oracle, scores1):
    """from y = theta, t = 1 the first step is ISTA's prox step (the momentum (t - 1) / t' is 0), and max_iter = 0
    changes nothing"""
    O = oracle
    rm, y, lam = scores1
    theta0 = np.array([0.3, 0.01, -0.02])
    res = A.proxgrad_accel(rm, y, theta0, lam=lam, epsilon_loss=0.0, max_iter=1)
    th, it, _ = O.proxgrad(rm, y, theta0, lam=lam, epsilon_loss=0.0, max_iter=1)
    assert res["iters"] == it == 1 and np.array_equal(res["theta"], th) and np.array_equal(res["y"], th)
    assert res["t"] == (1.0 + np.sqrt(5.0)) / 2.0 and res["restarts"] == 0
    res = A.proxgrad_accel(rm, y, theta0, lam=lam, max_iter=0)
    assert res["iters"] == 0 and np.array_equal(res["theta"], theta0) and np.array_equal(res["y"], theta0)


def test_slices_resume_exactly(oracle, scores1):
    """theta, y, t and the hook state carried between calls give one long call's iterates bit for bit"""
    rm, y, lam = scores1
    hook = [float("nan"), float("nan")]
    one = A.proxgrad_accel(rm, y, np.zeros(3), lam=lam, epsilon_loss=1e-300, max_iter=90, hook=hook)
    th, yy, t, hk, total, rs = np.zeros(3), None, 1.0, [float("nan"), float("nan")], 0, 0
    for _ in range(9):
        r = A.proxgrad_accel(rm, y, th, y=yy, t=t, lam=lam, epsilon_loss=1e-300, max_iter=10, hook=hk)
        th, yy, t, total, rs = r["theta"], r["y"], r["t"], total + r["iters"], rs + r["restarts"]
    assert total == one["iters"] == 90 and rs == one["restarts"]
    assert np.array_equal(th, one["theta"]) and np.array_equal(yy, one["y"]) and t == one["t"]
    assert hk == hook


def test_c2_sample_first_epochs_below_ista(oracle):
    """a C2-shaped sample (1 000 + 1 000 x 500 bp, k = 1..8 revcomp), the first epoch at N = 10 and 25: a few hundred
    iterations against thousands for ISTA, and a lower objective at the delta-loss stop"""
    from kmerlr_b200 import synth
    O = oracle
    buf, off, y = synth.training_set(1000, 1000, 500)
    ref = O.extract(O.make_config(1, 8, revcomp=True), (buf, off), threads=0)
    for N in (10, 25):
        r = O.select(ref, y, (1, 1), N, 0.0, [], [], tie=O.TIE_INDEX)
        sel = np.nonzero(r["mask"])[0]
        rm, lam = O.reduce(ref, sel), r["lam"]
        a = A.proxgrad_accel(rm, y, np.zeros(len(sel)), lam=lam, epsilon_loss=1e-8, max_iter=200000)
        th, it, _ = O.proxgrad(rm, y, np.zeros(len(sel)), lam=lam, epsilon_loss=1e-8, max_iter=200000)
        assert a["iters"] < it / 10 and a["restarts"] >= 1, (N, a["iters"], it)
        assert O.loss(rm, y, a["theta"], lam=lam) < O.loss(rm, y, th, lam=lam)
