"""kmerlr_proxgrad_accel (FISTA with gradient restart on reduced matrices, one GPU) against the restatement in
tests/accel_oracle.py: iteration by iteration, under every order-only tunable, in slices, on the leapfrog path, and
its refusals.  Needs a B200."""
import ctypes as C

import numpy as np
import pytest

import accel_oracle as A

pytestmark = pytest.mark.gpu

NAN2 = (float("nan"), float("nan"))


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def accel(K, d, theta, y=None, t=1.0, cw=(1.0, 1.0), lam=0.0, eps=0.0, eps_loss=0.0, cap=100, hook=None):
    """one kmerlr_proxgrad_accel call -> dict(theta, y, t, iters, restarts, delta, hook)"""
    from kmerlr_b200 import _lib
    theta = np.array(theta, dtype=np.float64)
    y = theta.copy() if y is None else np.array(y, dtype=np.float64)
    hk = np.array(NAN2 if hook is None else hook, dtype=np.float64)
    cwa = np.ascontiguousarray(cw, dtype=np.float64)
    tt, it, delta, rs = C.c_double(t), C.c_int64(), C.c_double(), C.c_int64()
    _lib.check(_lib.lib().kmerlr_proxgrad_accel(d.h, _p(theta), _p(y), tt, len(theta), _p(cwa), float(lam), 0.0, 1.0,
                                                eps, eps_loss, cap, _p(hk), it, delta, rs))
    return dict(theta=theta, y=y, t=tt.value, iters=it.value, restarts=rs.value, delta=delta.value, hook=hk)


def compare_with_oracle(r, o):
    assert r["iters"] == o["iters"], (r["iters"], o["iters"])
    assert r["restarts"] == o["restarts"], (r["restarts"], o["restarts"])
    assert np.max(np.abs(r["theta"] - o["theta"])) <= 1e-9
    assert np.array_equal(r["theta"] == 0.0, o["theta"] == 0.0)
    assert np.max(np.abs(r["y"] - o["y"])) <= 1e-9
    assert abs(r["delta"] - o["delta"]) <= 1e-6 * max(abs(o["delta"]), 1e-300)


def synthetic_reduced(K, O, n_fg, n_bg, L, N, sel_of):
    from kmerlr_b200 import synth
    buf, off, y = synth.training_set(n_fg, n_bg, L)
    kc, oc = K.NewKmerCounter(1, N, revcomp=True), O.make_config(1, N, revcomp=True)
    d = K.compile_test_data(None, kc, None, None, True, False, (buf, off))
    sel = sel_of(d.m)
    rd = K.select_data(d, sel)
    rd.SetLabels(y)
    d.free()
    return rd, O.reduce(O.extract(oc, (buf, off)), sel), y, sel


# ---------------------------------------------------------------------------------------------------
# iteration by iteration against the restatement
# ---------------------------------------------------------------------------------------------------
def test_matches_oracle_iteration_by_iteration(K, oracle, fixtures):
    """the 300 + 300 synthetic set of the ISTA test cut to 40 columns, and the TestScores1 reduction: stops by Epsilon,
    by EpsilonLoss and by max_iter (0 and 1 included) at the same iteration, with the same restarts"""
    O = oracle
    rd, rm, y, sel = synthetic_reduced(K, O, 300, 300, 200, 5,
                                       lambda m: np.unique(np.concatenate([[0], np.linspace(1, m, 40).astype(np.int64)])))
    X = np.vstack([fixtures["scoresLr_test_fg"], fixtures["scoresLr_test_bg"]])
    ys = np.array([1] * 8 + [0] * 8, dtype=np.uint8)
    ds = K.from_dense(X[:, [1, 6]])
    ds.SetLabels(ys)
    rs = O.from_dense(X[:, [1, 6]])
    lam1 = O.select(O.from_dense(X), ys, (1, 1), 2, 0.0, [], [], tie=O.TIE_GO118)["lam"]
    cw = np.array([0.9, 1.2])
    restarts = 0
    try:
        for d, ref, lab, w, cases in [
            (rd, rm, y, cw, [(0.0, 1e-7, 0.002, 5000), (1e-4, 0.0, 0.0005, 5000), (0.0, 1e-300, 0.001, 37),
                             (0.0, 0.0, 0.001, 0), (0.0, 0.0, 0.001, 1), (1e-6, 1e-10, 0.0, 5000)]),
            (ds, rs, ys, np.ones(2), [(0.0, 1e-13, lam1, 100000), (0.0, 1e-8, lam1, 100000), (1e-6, 0.0, lam1, 100000),
                                      (0.0, 0.0, lam1, 0), (0.0, 0.0, lam1, 1), (0.0, 0.0, lam1, 300)])]:
            for eps, eps_loss, lam, cap in cases:
                r = accel(K, d, np.zeros(ref.m + 1), cw=w, lam=lam, eps=eps, eps_loss=eps_loss, cap=cap)
                o = A.proxgrad_accel(ref, lab, np.zeros(ref.m + 1), cw=tuple(w), lam=lam, epsilon=eps,
                                     epsilon_loss=eps_loss, max_iter=cap)
                compare_with_oracle(r, o)
                assert r["t"] == o["t"]
                if cap in (0, 1, 37, 300):
                    assert r["iters"] == cap
                restarts += r["restarts"]
        assert restarts > 0
    finally:
        rd.free(); ds.free()


# ---------------------------------------------------------------------------------------------------
# order-only tunables
# ---------------------------------------------------------------------------------------------------
TUNABLES = [(pe, sl, bps) for pe in (0, 1) for sl in (0, 1, 2) for bps in (0, 2)]


def test_tunables_only_change_the_order(K, oracle):
    """persistent x small_long x persist_bps on counts and real values (Transform-scaled), short rows and long rows (the
    matrices of the ISTA long-row test): theta, y, t, iterations, restarts, delta and the hook state bit for bit"""
    O = oracle
    short, _, ys, sels = synthetic_reduced(K, O, 700, 650, 150, 6,
                                           lambda m: np.unique(np.concatenate([[0], np.linspace(1, m, 40).astype(np.int64)])))
    long_, _, yl, sell = synthetic_reduced(K, O, 900, 833, 180, 6, lambda m: np.unique(np.concatenate(
        [[0], np.arange(1, 45), np.linspace(50, m, 30).astype(np.int64)])))
    assert long_.nnz >= 30 * long_.n
    mats = [short, long_]
    for d, lab, sel in ((short, ys, sels), (long_, yl, sell)):
        sc = K.Transform(Scale=np.concatenate([[1.0], 1.0 / (1.0 + np.arange(len(sel) - 1) % 7)])).Apply(d)
        sc.SetLabels(lab)
        mats.append(sc)
    cw = (0.8, 1.3)
    try:
        for d in mats:
            for eps, eps_loss, lam, cap in [(0.0, 0.0, 1e-3, 61), (1e-6, 0.0, 1e-3, 20000), (0.0, 1e-9, 2e-3, 20000),
                                            (0.0, 0.0, 1e-3, 0)]:
                first = None
                for t in TUNABLES:
                    K.option("persistent", t[0]); K.option("small_long", t[1]); K.option("persist_bps", t[2])
                    r = accel(K, d, np.zeros(d.m + 1), cw=cw, lam=lam, eps=eps, eps_loss=eps_loss, cap=cap)
                    if first is None:
                        first = (t, r)
                        continue
                    f = first[1]
                    what = (t, first[0], eps, eps_loss, cap)
                    for k in ("iters", "restarts", "t"):
                        assert r[k] == f[k], (k, what, r[k], f[k])
                    assert r["delta"] == f["delta"] or (np.isnan(r["delta"]) and np.isnan(f["delta"])), what
                    for k in ("theta", "y", "hook"):
                        assert np.array_equal(r[k], f[k], equal_nan=True), (k, what)
                if cap == 61:
                    assert first[1]["iters"] == 61
    finally:
        K.option("persistent", 1); K.option("small_long", -1); K.option("persist_bps", 0)
        for d in mats:
            d.free()


# ---------------------------------------------------------------------------------------------------
# resumable in slices
# ---------------------------------------------------------------------------------------------------
def test_resumable_in_slices(K, oracle):
    """KmerLrEstimator(Accelerated=True) run in slices of k iterations (theta, y, t and hook_state carried between the
    calls on the same reduced data) gives one long call's results bit for bit, also when the loss stop falls inside a
    slice"""
    rd, _, _, _ = synthetic_reduced(K, oracle, 400, 400, 150, 6,
                                    lambda m: np.unique(np.concatenate([[0], np.linspace(1, m, 30).astype(np.int64)])))
    try:
        for eps_loss, cap, k in ((1e-300, 60, 10), (1e-9, 100000, 7)):
            one = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=eps_loss, MaxIterations=cap, Accelerated=True)
            one.Theta = np.zeros(rd.m + 1)
            it1, d1 = one.estimate_proximal(rd, 1e-3)
            sl = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=eps_loss, MaxIterations=k, Accelerated=True)
            sl.Theta = np.zeros(rd.m + 1)
            total = restarts = 0
            while total < cap:
                it, delta = sl.estimate_proximal(rd, 1e-3)
                total += it
                restarts += sl.accel_state[3]
                if it < k:
                    break
            assert total == it1 and (it1 == 60 if cap == 60 else 0 < it1 < cap), (it1, total)
            assert restarts == one.accel_state[3]
            assert np.array_equal(one.Theta, sl.Theta)
            assert np.array_equal(one.accel_state[1], sl.accel_state[1]) and one.accel_state[2] == sl.accel_state[2]
            assert np.array_equal(one.hook_state, sl.hook_state)
            assert delta == d1
    finally:
        rd.free()


# ---------------------------------------------------------------------------------------------------
# the leapfrog path
# ---------------------------------------------------------------------------------------------------
def test_leapfrog_path_on_a_c2_shaped_sample(K, oracle):
    """2 000 sequences x 500 bp, k = 1..8 revcomp, --lambda-auto=5,10 with Accelerated=True: the restatement's epochs,
    lambda sequence and selected sets, iterations within 1, theta within 1e-5; the first lambda is ISTA's bit for bit
    (a function of g(0) alone); the first epochs at N = 10 and 25 end at a lower objective than ISTA's"""
    from kmerlr_b200 import synth
    O = oracle
    buf, off, y = synth.training_set(1000, 1000, 500)
    kc, oc = K.NewKmerCounter(1, 8, revcomp=True), O.make_config(1, 8, revcomp=True)
    d = K.compile_test_data(None, kc, None, None, True, False, (buf, off))
    d.SetLabels(y)
    ref = O.extract(oc, (buf, off), threads=0)
    try:
        est = K.KmerLrEstimator(EpsilonLoss=1e-8, tie=K.TIE_INDEX, MaxIterations=200000, Accelerated=True)
        oest = A.EstimatorState()
        for N in (5, 10):
            est.path = []
            est.estimate_loop(d, N)
            res = A.estimate_loop(ref, y, (1, 1), N, oest, tie=O.TIE_INDEX, epsilon_loss=1e-8, max_iter=200000)
            assert len(est.path) == res["epochs"] and res["epochs"] >= 1
            assert np.array_equal(est.active_idx, oest.active_idx)
            lams = np.array([p[0] for p in est.path])
            assert np.allclose(lams, res["lambdas"], rtol=1e-9, atol=0)
            its = np.array([p[1] for p in est.path])
            assert np.all(np.abs(its - np.array(res["iters"])) <= 1), (its, res["iters"])
            assert np.max(np.abs(est.Theta - oest.active_theta)) <= 1e-5 * max(1.0, np.max(np.abs(oest.active_theta)))
        for N in (10, 25):
            runs = {}
            for acc in (False, True):
                e = K.KmerLrEstimator(EpsilonLoss=1e-8, tie=K.TIE_INDEX, MaxIterations=200000, MaxEpochs=1, Accelerated=acc)
                e.estimate_loop(d, N)
                sel = np.concatenate([[0], e.active_idx])
                runs[acc] = (e.path[0][0], e.path[0][1], O.loss(O.reduce(ref, sel), y, e.Theta, (1, 1), e.path[0][0]), sel)
            assert runs[True][0] == runs[False][0]                      # the first lambda, bit for bit
            assert np.array_equal(runs[True][3], runs[False][3])
            assert runs[True][2] < runs[False][2], (N, runs)
            assert runs[True][1] < runs[False][1] / 5, (N, runs)
    finally:
        d.free()


# ---------------------------------------------------------------------------------------------------
# refusals
# ---------------------------------------------------------------------------------------------------
def test_refusals(K, oracle):
    """KMERLR_ERR_ARG with a message: more than 1023 columns, a matrix-free view, t < 1 or not finite, null y or t.
    (A sharded matrix is refused too; that needs more than one rank and is not exercised here.)"""
    from kmerlr_b200 import _lib, synth
    L = _lib.lib()
    rng = np.random.default_rng(5)
    n = 64
    big = K.from_dense(rng.integers(0, 3, size=(n, 1024)).astype(np.float64))
    lab = (rng.random(n) < 0.5).astype(np.uint8)
    lab[0], lab[1] = 1, 0
    big.SetLabels(lab)
    buf, off, y = synth.training_set(50, 50, 100)
    mf = K.compile_test_data(None, K.NewKmerCounter(1, 3, revcomp=True), None, None, True, False, (buf, off))
    mf.SetLabels(y)
    small = K.select_data(mf, np.arange(0, 11))
    small.SetLabels(y)
    try:
        assert mf.m + 1 <= 1024

        def refused(d, match, **kw):
            with pytest.raises(K.KmerLrError) as e:
                accel(K, d, np.zeros(d.m + 1), lam=1e-3, cap=5, **kw)
            assert e.value.code == _lib.ERR_ARG and match in str(e.value), str(e.value)

        refused(big, "reduced matrices only")
        refused(mf, "reduced matrices only")
        for t in (0.5, 0.0, -1.0, float("nan"), float("inf")):
            refused(small, "momentum t", t=t)
        theta, y0, cw, hk = np.zeros(small.m + 1), np.zeros(small.m + 1), np.ones(2), np.array(NAN2)
        it, delta, rs, tt = C.c_int64(), C.c_double(), C.c_int64(), C.c_double(1.0)
        for yp, tp in ((None, tt), (_p(y0), None)):
            rc = L.kmerlr_proxgrad_accel(small.h, _p(theta), yp, tp, len(theta), _p(cw), 1e-3, 0.0, 1.0, 0.0, 0.0, 5,
                                         _p(hk), it, delta, rs)
            assert rc == _lib.ERR_ARG and b"null argument" in L.kmerlr_last_error()
        # a reduced matrix of the same data is accepted, and ISTA still takes the matrix-free view
        assert accel(K, small, np.zeros(small.m + 1), lam=1e-3, cap=5)["iters"] == 5
        est = K.KmerLrEstimator(EpsilonLoss=0.0, MaxIterations=3)
        est.Theta = np.zeros(mf.m + 1)
        assert est.estimate_proximal(mf, 1e-3)[0] == 3
    finally:
        big.free(); small.free(); mf.free()
