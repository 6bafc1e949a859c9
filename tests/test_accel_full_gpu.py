"""kmerlr_proxgrad_accel_full (FISTA with gradient restart on every one-GPU matrix) against the restatement in
tests/accel_oracle.py: matrices straight from the extraction (matrix-free and stored rows, counts and binarized),
imported, scaled, row subsets and wide reduced matrices; the same bits as kmerlr_proxgrad_accel on reduced matrices;
determinism, slices, the estimator, the launch budget and the refusals.  Needs a B200."""
import contextlib
import ctypes as C

import numpy as np
import pytest

import accel_oracle as A

pytestmark = pytest.mark.gpu

NAN2 = (float("nan"), float("nan"))
CW = (0.9, 1.2)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def accel(K, d, theta, y=None, t=1.0, cw=(1.0, 1.0), lam=0.0, eps=0.0, eps_loss=0.0, cap=100, hook=None,
          entry="kmerlr_proxgrad_accel_full"):
    """one call of `entry` -> dict(theta, y, t, iters, restarts, delta, hook)"""
    from kmerlr_b200 import _lib
    theta = np.array(theta, dtype=np.float64)
    y = theta.copy() if y is None else np.array(y, dtype=np.float64)
    hk = np.array(NAN2 if hook is None else hook, dtype=np.float64)
    cwa = np.ascontiguousarray(cw, dtype=np.float64)
    tt, it, delta, rs = C.c_double(t), C.c_int64(), C.c_double(), C.c_int64()
    _lib.check(getattr(_lib.lib(), entry)(d.h, _p(theta), _p(y), tt, len(theta), _p(cwa), float(lam), 0.0, 1.0, eps,
                                          eps_loss, cap, _p(hk), it, delta, rs))
    return dict(theta=theta, y=y, t=tt.value, iters=it.value, restarts=rs.value, delta=delta.value, hook=hk)


def compare_with_oracle(r, o, what=None):
    assert r["iters"] == o["iters"], (what, r["iters"], o["iters"])
    assert r["restarts"] == o["restarts"], (what, r["restarts"], o["restarts"])
    assert np.max(np.abs(r["theta"] - o["theta"])) <= 1e-9, what
    assert np.array_equal(r["theta"] == 0.0, o["theta"] == 0.0), what
    assert np.max(np.abs(r["y"] - o["y"])) <= 1e-9, what
    assert abs(r["delta"] - o["delta"]) <= 1e-6 * max(abs(o["delta"]), 1e-300), what
    assert r["t"] == o["t"], what


def dense_of(d):
    """the rows of a device matrix read back, as a dense array"""
    rp, col, val = d.rows()
    X = np.zeros((d.n, d.m))
    X[np.repeat(np.arange(d.n), np.diff(rp)), col] = val
    return X


def first_lambda(O, ref, y, N=10):
    """the lambda of the first leapfrog selection at theta = 0 (unit class weights, as estimate_loop without balance),
    moved off the value of the gradient it is taken from: at exactly that lambda the first prox step from theta = 0
    leaves one coefficient on the threshold, where a last-bit difference decides whether it is zero"""
    return O.select(ref, y, (1.0, 1.0), N, 0.0, [], [], tie=O.TIE_INDEX)["lam"] * (1.0 + 1e-6)


@pytest.fixture(scope="module")
def sample(K, oracle):
    """300 + 300 sequences x 200 bp, k = 1..6 revcomp (2 772 columns): the count matrix and its oracle twin"""
    from kmerlr_b200 import synth
    buf, off, y = synth.training_set(300, 300, 200)
    d = K.compile_test_data(None, K.NewKmerCounter(1, 6, revcomp=True), None, None, True, False, (buf, off))
    d.SetLabels(y)
    ref = oracle.extract(oracle.make_config(1, 6, revcomp=True), (buf, off))
    assert d.m == ref.m and d.m > 1023
    yield dict(buf=buf, off=off, y=y, d=d, ref=ref)
    d.free()


@contextlib.contextmanager
def stored_rows(K, on):
    """on: the pass over the stored rows in place of the matrix-free pass (kmerlr_option("implicit", 0))"""
    K.option("implicit", 0 if on else 1)
    try:
        yield
    finally:
        K.option("implicit", 1)


# ---------------------------------------------------------------------------------------------------
# iteration by iteration against the restatement
# ---------------------------------------------------------------------------------------------------
def test_matches_oracle_iteration_by_iteration(K, oracle, sample):
    """counts matrix-free and on stored rows, binarized (repeat events), an imported dense matrix of 1 500 columns, a
    Transform(Scale=...) of the counts and a row subset: stops by Epsilon, by EpsilonLoss and by max_iter (0, 1 and a
    mid-run cap) at the same iteration with the same restarts, unequal class weights"""
    from kmerlr_b200 import synth
    O = oracle
    d, ref, y = sample["d"], sample["ref"], sample["y"]
    owned = []
    buf, off, yb = synth.training_set(250, 250, 200)
    db = K.compile_test_data(None, K.NewKmerCounter(1, 6, revcomp=True), None, None, True, True, (buf, off))
    db.SetLabels(yb)
    owned.append(db)
    refb = O.extract(O.make_config(1, 6, revcomp=True, binarize=True), (buf, off))
    rng = np.random.default_rng(11)
    X = rng.integers(0, 4, size=(400, 1500)).astype(np.float64) * (rng.random((400, 1500)) < 0.05)
    yd = (rng.random(400) < 0.5).astype(np.uint8)
    X[yd == 1, :40] += rng.integers(0, 2, size=(int(yd.sum()), 40))
    dd = K.from_dense(X)
    dd.SetLabels(yd)
    owned.append(dd)
    sc = K.Transform(Scale=np.concatenate([[1.0], 1.0 / (1.0 + np.arange(d.m) % 5)])).Apply(d)
    sc.SetLabels(y)
    owned.append(sc)
    rows = np.concatenate([np.arange(0, 600, 3), np.arange(1, 600, 3)])
    sub = d.subset(rows)
    owned.append(sub)
    cases = [(0.0, 1e-9, 3000), (1e-6, 0.0, 3000), (0.0, 0.0, 0), (0.0, 0.0, 1), (0.0, 0.0, 37)]
    mats = [("counts, matrix-free", d, ref, y, False), ("counts, stored rows", d, ref, y, True),
            ("binarized", db, refb, yb, False), ("imported dense", dd, O.from_dense(X), yd, False),
            ("scaled", sc, O.from_dense(dense_of(sc)), y, False),
            ("row subset", sub, O.from_dense(dense_of(sub)), y[rows], False)]
    restarts = 0
    try:
        assert db.m > 1023 and sc.m == d.m and sub.m == d.m
        for name, dev, oref, lab, stored in mats:
            lam = first_lambda(O, oref, lab)
            for eps, eps_loss, cap in cases:
                with stored_rows(K, stored):
                    r = accel(K, dev, np.zeros(dev.m + 1), cw=CW, lam=lam, eps=eps, eps_loss=eps_loss, cap=cap)
                o = A.proxgrad_accel(oref, lab, np.zeros(oref.m + 1), cw=CW, lam=lam, epsilon=eps, epsilon_loss=eps_loss,
                                     max_iter=cap)
                compare_with_oracle(r, o, (name, eps, eps_loss, cap))
                if eps == 0.0 and eps_loss == 0.0:
                    assert r["iters"] == cap
                else:
                    assert np.any(r["theta"][1:] != 0.0), name
                restarts += r["restarts"]
        assert restarts > 0
    finally:
        for m in owned:
            m.free()


def test_matrix_free_iterations_equal_stored_row_iterations(K, sample):
    """a few accelerated iterations through the matrix-free pass and through the stored rows agree within the bars the
    ISTA version of this test holds"""
    d = sample["d"]
    runs = []
    for stored in (False, True):
        with stored_rows(K, stored):
            runs.append(accel(K, d, np.zeros(d.m + 1), cw=CW, lam=1e-3, eps_loss=1e-300, cap=6))
    a, b = runs
    assert np.any(a["theta"][1:] != 0.0)
    for k in ("theta", "y"):
        assert np.max(np.abs(a[k] - b[k])) <= 1e-13 * max(np.max(np.abs(b[k])), 1e-300), k
    assert np.all(np.isfinite(a["hook"])) and np.allclose(a["hook"], b["hook"], rtol=1e-13, atol=0.0)
    assert a["iters"] == b["iters"] == 6 and a["restarts"] == b["restarts"] and a["t"] == b["t"]


# ---------------------------------------------------------------------------------------------------
# reduced matrices: the body of kmerlr_proxgrad_accel
# ---------------------------------------------------------------------------------------------------
def test_same_body_on_reduced_matrices(K, sample):
    """short and long reduced rows, persistent 0 and 1: kmerlr_proxgrad_accel_full gives kmerlr_proxgrad_accel's bits"""
    d, y = sample["d"], sample["y"]
    mats = []
    for sel in (np.unique(np.concatenate([[0], np.linspace(1, d.m, 40).astype(np.int64)])), np.arange(0, 80)):
        r = K.select_data(d, sel)
        r.SetLabels(y)
        mats.append(r)
    assert mats[1].nnz >= 8 * mats[1].n
    try:
        for pe in (0, 1):
            K.option("persistent", pe)
            for rd in mats:
                for eps, eps_loss, cap in ((0.0, 0.0, 45), (1e-6, 0.0, 20000), (0.0, 1e-9, 20000)):
                    a, b = [accel(K, rd, np.zeros(rd.m + 1), cw=CW, lam=1e-3, eps=eps, eps_loss=eps_loss, cap=cap,
                                  entry=e) for e in ("kmerlr_proxgrad_accel_full", "kmerlr_proxgrad_accel")]
                    what = (pe, rd.m, eps, eps_loss, cap)
                    for k in ("iters", "restarts", "t"):
                        assert a[k] == b[k], (k, what)
                    assert a["delta"] == b["delta"] or (np.isnan(a["delta"]) and np.isnan(b["delta"])), what
                    for k in ("theta", "y", "hook"):
                        assert np.array_equal(a[k], b[k], equal_nan=True), (k, what)
    finally:
        K.option("persistent", 1)
        for m in mats:
            m.free()


# ---------------------------------------------------------------------------------------------------
# determinism and slices
# ---------------------------------------------------------------------------------------------------
def test_deterministic_and_resumable_in_slices(K, oracle, sample):
    """the same full-space call twice gives the same bits; KmerLrEstimator(Accelerated=True) in slices of k iterations
    (theta, y, t and hook_state carried) gives one long call's iterates and stopping point bit for bit"""
    d, ref, y = sample["d"], sample["ref"], sample["y"]
    lam = first_lambda(oracle, ref, y)
    a, b = [accel(K, d, np.zeros(d.m + 1), lam=lam, eps_loss=1e-9, cap=5000) for _ in range(2)]
    for k in ("iters", "restarts", "t", "delta"):
        assert a[k] == b[k], k
    for k in ("theta", "y", "hook"):
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    for eps_loss, cap, k in ((1e-300, 60, 10), (1e-9, 100000, 7)):
        one = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=eps_loss, MaxIterations=cap, Accelerated=True)
        one.Theta = np.zeros(d.m + 1)
        it1, d1 = one.estimate_proximal(d, lam)
        sl = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=eps_loss, MaxIterations=k, Accelerated=True)
        sl.Theta = np.zeros(d.m + 1)
        total = restarts = 0
        while total < cap:
            it, delta = sl.estimate_proximal(d, lam)
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


# ---------------------------------------------------------------------------------------------------
# the estimator
# ---------------------------------------------------------------------------------------------------
def test_estimate_proximal_on_the_full_matrix(K, oracle, sample):
    """the fixed-lambda fit: KmerLrEstimator(Accelerated=True).estimate_proximal on the whole feature space equals the
    restatement"""
    d, ref, y = sample["d"], sample["ref"], sample["y"]
    lam = first_lambda(oracle, ref, y)
    est = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=1e-9, MaxIterations=20000, Accelerated=True)
    est.Theta = np.zeros(d.m + 1)
    est.ClassWeights = np.array(CW)
    it, delta = est.estimate_proximal(d, lam)
    o = A.proxgrad_accel(ref, y, np.zeros(d.m + 1), cw=CW, lam=lam, epsilon_loss=1e-9, max_iter=20000)
    compare_with_oracle(dict(theta=est.Theta, y=est.accel_state[1], t=est.accel_state[2], iters=it,
                             restarts=est.accel_state[3], delta=delta), o)
    assert 0 < it < 20000 and np.count_nonzero(est.Theta[1:]) > 0


def test_leapfrog_epochs_on_wide_reduced_matrices(K, oracle, sample):
    """--lambda-auto=1100: two epochs whose reduced matrices have more than 1 023 columns; every epoch equals the
    restatement on the oracle's reduction of the same selection, from the same start (theta, hook state; y = theta,
    t = 1): iterations, restarts, theta, y, t and the objective.  The epochs are capped at 400 iterations: near the
    optimum the restart test compares a dot product of two vanishing steps with 0, and last-bit differences of the
    gradient then decide it either way (the two runs still converge, at different iteration counts)"""
    d, ref, y = sample["d"], sample["ref"], sample["y"]
    est = K.KmerLrEstimator(EpsilonLoss=1e-8, tie=K.TIE_INDEX, MaxIterations=400, MaxEpochs=2, Accelerated=True)
    epochs = []
    solve = est.estimate_proximal

    def logged(reduced, lam):
        start = (np.concatenate([[0], est.active_idx]), est.Theta.copy(), list(est.hook_state), lam, reduced.m)
        it, delta = solve(reduced, lam)
        epochs.append((start, dict(theta=est.Theta.copy(), y=est.accel_state[1].copy(), t=est.accel_state[2], iters=it,
                                   restarts=est.accel_state[3], delta=delta)))
        return it, delta

    est.estimate_proximal = logged
    est.estimate_loop(d, 1100)
    assert len(epochs) == 2
    for (sel, th0, hook, lam, m), r in epochs:
        assert m + 1 > 1024 and len(sel) == m + 1
        rm = oracle.reduce(ref, sel)
        o = A.proxgrad_accel(rm, y, th0, lam=lam, epsilon_loss=1e-8, max_iter=400, hook=hook)
        compare_with_oracle(r, o, m)
        f, fo = (oracle.loss(rm, y, x, (1.0, 1.0), lam) for x in (r["theta"], o["theta"]))
        assert abs(f - fo) <= 1e-9 * abs(fo)


# ---------------------------------------------------------------------------------------------------
# launch budget
# ---------------------------------------------------------------------------------------------------
def test_one_launch_more_than_an_ista_step(K, sample):
    """one accelerated prox step on the full feature space costs one launch more than an ISTA step (the momentum
    kernel), matrix-free and on stored rows"""
    from kmerlr_b200 import _lib
    d = sample["d"]
    cwa, hk = np.ones(2), np.array(NAN2)
    it, delta = C.c_int64(), C.c_double()

    def launches(acc, cap):
        n0 = K.launch_count()
        if acc:
            accel(K, d, np.zeros(d.m + 1), lam=1e-3, cap=cap)
        else:
            th = np.zeros(d.m + 1)
            _lib.check(_lib.lib().kmerlr_proxgrad(d.h, _p(th), len(th), _p(cwa), 1e-3, 0.0, 1.0, 0.0, 0.0, cap, _p(hk),
                                                  it, delta))
        return K.launch_count() - n0

    for stored in (False, True):
        with stored_rows(K, stored):
            launches(False, 1), launches(True, 1)          # whatever a first call on the view sets up
            per = {acc: launches(acc, 4) - launches(acc, 3) for acc in (False, True)}
        assert per[False] > 0 and per[True] == per[False] + 1, (stored, per)


# ---------------------------------------------------------------------------------------------------
# refusals
# ---------------------------------------------------------------------------------------------------
def test_refusals(K, sample):
    """KMERLR_ERR_ARG with a message: t < 1 or not finite, a null theta, y, t or class_w, a matrix without labels, an
    empty set.  (A sharded matrix is refused too; that needs more than one rank and is not exercised here.)"""
    from kmerlr_b200 import _lib
    L = _lib.lib()
    d = sample["d"]
    nolab = K.from_dense(np.eye(4))
    empty = K.from_dense(np.zeros((0, 5)))
    empty.SetLabels(np.zeros(0, dtype=np.uint8))
    try:
        def refused(m, match, **kw):
            with pytest.raises(K.KmerLrError) as e:
                accel(K, m, np.zeros(m.m + 1), lam=1e-3, cap=5, **kw)
            assert e.value.code == _lib.ERR_ARG and match in str(e.value), str(e.value)

        for t in (0.5, 0.0, -1.0, float("nan"), float("inf")):
            refused(d, "momentum t", t=t)
        refused(nolab, "no labels")
        refused(empty, "empty data set")
        theta, y0, cw, hk = np.zeros(d.m + 1), np.zeros(d.m + 1), np.ones(2), np.array(NAN2)
        it, delta, rs, tt = C.c_int64(), C.c_double(), C.c_int64(), C.c_double(1.0)
        for tp, yp, tq, cp in ((None, _p(y0), tt, _p(cw)), (_p(theta), None, tt, _p(cw)), (_p(theta), _p(y0), None, _p(cw)),
                               (_p(theta), _p(y0), tt, None)):
            rc = L.kmerlr_proxgrad_accel_full(d.h, tp, yp, tq, len(theta), cp, 1e-3, 0.0, 1.0, 0.0, 0.0, 5, _p(hk), it,
                                              delta, rs)
            assert rc == _lib.ERR_ARG and b"null argument" in L.kmerlr_last_error()
        # the matrix-free view and more than 1023 columns are taken
        assert accel(K, d, np.zeros(d.m + 1), lam=1e-3, cap=5)["iters"] == 5
    finally:
        nolab.free(); empty.free()
