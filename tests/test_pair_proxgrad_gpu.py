"""Fixed-lambda fits over the pair-feature space: kmerlr_step_size_pairs, kmerlr_proxgrad_pairs and
kmerlr_proxgrad_pairs_accel on the raw matrix against the explicit expansion kmerlr_reduce(h, 0 .. Dim-1), its CPU
oracle twin O.reduce(mat, arange(Dim)) and the restatements O.proxgrad / accel_oracle.proxgrad_accel; the device-built
pair-term list on both sides of PAIR_TERMS_MAX; m <= 44 (Dim <= 1 024, where the reduced-matrix kernels must not run)
and m = 1; slices and determinism; C4 scale against a dense fp64 restatement on the device; the launch budget; the
refusals.  Needs a B200."""
import ctypes as C

import numpy as np
import pytest

import accel_oracle as A

pytestmark = pytest.mark.gpu

NAN2 = (float("nan"), float("nan"))
CW = (0.9, 1.2)
ULP = 2.0 ** -52


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def coeff_dim(m):
    return (m + 1) * m // 2 + 1


def ista(K, d, theta, cw=(1.0, 1.0), lam=0.0, eps=0.0, eps_loss=0.0, cap=100, hook=None, step_factor=1.0,
         entry="kmerlr_proxgrad_pairs"):
    """one call of kmerlr_proxgrad_pairs (or kmerlr_proxgrad) -> dict(theta, iters, delta, hook)"""
    from kmerlr_b200 import _lib
    theta = np.array(theta, dtype=np.float64)
    hk = np.array(NAN2 if hook is None else hook, dtype=np.float64)
    cwa = np.ascontiguousarray(cw, dtype=np.float64)
    it, delta = C.c_int64(), C.c_double()
    _lib.check(getattr(_lib.lib(), entry)(d.h, _p(theta), len(theta), _p(cwa), float(lam), 0.0, step_factor, eps,
                                          eps_loss, cap, _p(hk), it, delta))
    return dict(theta=theta, iters=it.value, delta=delta.value, hook=hk)


def fista(K, d, theta, y=None, t=1.0, cw=(1.0, 1.0), lam=0.0, eps=0.0, eps_loss=0.0, cap=100, hook=None,
          entry="kmerlr_proxgrad_pairs_accel"):
    """one call of kmerlr_proxgrad_pairs_accel (or kmerlr_proxgrad_accel_full) -> dict(theta, y, t, iters, restarts,
    delta, hook)"""
    from kmerlr_b200 import _lib
    theta = np.array(theta, dtype=np.float64)
    y = theta.copy() if y is None else np.array(y, dtype=np.float64)
    hk = np.array(NAN2 if hook is None else hook, dtype=np.float64)
    cwa = np.ascontiguousarray(cw, dtype=np.float64)
    tt, it, delta, rs = C.c_double(t), C.c_int64(), C.c_double(), C.c_int64()
    _lib.check(getattr(_lib.lib(), entry)(d.h, _p(theta), _p(y), tt, len(theta), _p(cwa), float(lam), 0.0, 1.0, eps,
                                          eps_loss, cap, _p(hk), it, delta, rs))
    return dict(theta=theta, y=y, t=tt.value, iters=it.value, restarts=rs.value, delta=delta.value, hook=hk)


def step_pairs(d):
    from kmerlr_b200 import _lib
    s = C.c_double()
    _lib.check(_lib.lib().kmerlr_step_size_pairs(d.h, 0.0, 1.0, s))
    return s.value


def step_plain(d):
    from kmerlr_b200 import _lib
    s = C.c_double()
    _lib.check(_lib.lib().kmerlr_step_size(d.h, 0.0, 1.0, s))
    return s.value


def close(a, b, bar=1e-9):
    return np.max(np.abs(a - b)) <= bar


def pair_lambda(O, ref, y, N=10):
    """the lambda of the first Select over the pair space at theta = 0, moved off the gradient value it comes from"""
    return O.select(ref, y, (1.0, 1.0), N, 0.0, [], [], cooccurrence=True, tie=O.TIE_INDEX)["lam"] * (1.0 + 1e-6)


def rows_of(d):
    rp, col, val = d.rows()
    return np.asarray(rp, dtype=np.int64), np.asarray(col), np.asarray(val, dtype=np.float64)


@pytest.fixture(scope="module")
def c1(K, oracle, fixtures):
    """the C1 fixtures (fg || bg) at k = 1..4 revcomp (m = 180, Dim = 16 291) as counts, binarized, f64 rows and a row
    subset; each with its oracle twin and the oracle's explicit expansion"""
    from conftest import cat
    O = oracle
    buf, off, y = cat(fixtures, "kmerLr_test_fg", "kmerLr_test_bg")
    nfg = int(y.sum())
    fg, bg = (buf[:off[nfg]], off[:nfg + 1]), (buf[off[nfg]:], off[nfg:] - off[nfg])
    out, owned = {}, []
    for kind, binz in (("counts", False), ("binarized", True)):
        d = K.compile_training_data(None, K.NewKmerCounter(1, 4, revcomp=True), None, None, True, binz, fg, bg)
        owned.append(d)
        ref = O.extract(O.make_config(1, 4, revcomp=True, binarize=binz), (buf, off))
        out[kind] = (d, ref, y)
    d = out["counts"][0]
    assert d.m == 180 and coeff_dim(d.m) == 16291
    rp, col, val = rows_of(d)
    f = K.from_csr(d.n, d.m, rp, col, val)
    f.SetLabels(y)
    owned.append(f)
    out["f64"] = (f, O.from_csr(d.n, d.m, rp, col, val), y)
    rows = np.array([0, 2, 3, 5, 8, 9, 11, 12, 14, 17, 19, 20, 21], dtype=np.int64)
    sub = d.subset(rows)
    owned.append(sub)
    srp, scol, sval = rows_of(sub)
    out["subset"] = (sub, O.from_csr(sub.n, sub.m, srp, scol, sval), y[rows])
    for kind in list(out):
        dd, ref, yy = out[kind]
        out[kind] = dict(d=dd, ref=ref, y=yy, exp=O.reduce(ref, np.arange(coeff_dim(ref.m))))
    yield out
    for h in owned:
        h.free()


# ---------------------------------------------------------------------------------------------------
# 1. step size of the pair-expanded rows
# ---------------------------------------------------------------------------------------------------
def test_step_size_is_the_explicit_expansions(K, oracle, fixtures, c1):
    """integer rows: the bits of the oracle's and the device's step size on the explicit expansion; f64 rows: within a
    few ulp.  C1 counts and binarized, TestKmers6 binarized (m = 70, Dim = 2 486), a synthetic matrix of large counts."""
    from conftest import cat
    O = oracle
    cases = [(c1["counts"]["d"], c1["counts"]["ref"]), (c1["binarized"]["d"], c1["binarized"]["ref"])]
    buf, off, y = cat(fixtures, "kmerLr_test_co_fg", "kmerLr_test_co_bg")
    nfg = int(y.sum())
    co = K.compile_training_data(None, K.NewKmerCounter(2, 6, revcomp=True), None, None, True, True,
                                 (buf[:off[nfg]], off[:nfg + 1]), (buf[off[nfg]:], off[nfg:] - off[nfg]))
    rng = np.random.default_rng(3)
    n, m = 50, 12
    X = rng.integers(0, 3000, size=(n, m)) * (rng.random((n, m)) < 0.5)
    X[0, :3] = [2900, 2950, 2999]
    rp = np.concatenate([[0], np.cumsum((X != 0).sum(1))]).astype(np.int64)
    col = np.nonzero(X)[1].astype(np.int32)
    big = K.from_csr(n, m, rp, col, X[X != 0].astype(np.float64))
    owned = [co, big]
    try:
        assert co.m == 70 and coeff_dim(co.m) == 2486
        cases.append((co, O.extract(O.make_config(2, 6, revcomp=True, binarize=True), (buf, off))))
        # counts up to 2 999 (exact integers in f64 rows): the expansion's row sums stay below 2^53, where both sides are
        # exact
        cases.append((big, O.from_csr(n, m, rp, col, X[X != 0].astype(np.float64))))
        for d, ref in cases:
            e = K.select_data(d, np.arange(coeff_dim(d.m)))
            owned.append(e)
            s = step_pairs(d)
            assert s == O.step_size(O.reduce(ref, np.arange(coeff_dim(ref.m)))), d.m
            assert s == step_plain(e), d.m
        # f64 rows: within a few ulp of the expansion's
        f = c1["f64"]["d"]
        e = K.select_data(f, np.arange(coeff_dim(f.m)))
        owned.append(e)
        assert abs(step_pairs(f) - step_plain(e)) <= 4 * ULP * step_plain(e)
        # the counts' value: S2 + (S2^2 - S4) / 2 of the largest row, restated
        rpc, colc, valc = rows_of(c1["counts"]["d"])
        nrm = max(np.sum(v ** 2) + (np.sum(v ** 2) ** 2 - np.sum(v ** 4)) / 2
                  for v in np.split(valc, rpc[1:-1]))
        assert step_pairs(c1["counts"]["d"]) == 1.0 / (2.0 * (0.25 * (nrm + 1.0)))
    finally:
        for h in owned:
            h.free()


# ---------------------------------------------------------------------------------------------------
# 2. - 3. ISTA and FISTA against the explicit expansion
# ---------------------------------------------------------------------------------------------------
CASES = [(0.0, 1e-9, 3000), (1e-6, 0.0, 3000), (0.0, 0.0, 0), (0.0, 0.0, 1), (0.0, 0.0, 37)]


@pytest.mark.parametrize("kind", ["counts", "binarized", "f64", "subset"])
def test_ista_matches_the_explicit_expansion(K, oracle, c1, kind):
    """stops by Epsilon, by EpsilonLoss and at max_iter 0, 1, 37: the oracle's iteration count and theta within 1e-9;
    kmerlr_proxgrad on kmerlr_reduce(all) too"""
    O = oracle
    c = c1[kind]
    d, y, exp = c["d"], c["y"], c["exp"]
    nt = coeff_dim(d.m)
    lam = pair_lambda(O, c["ref"], y)
    e = K.select_data(d, np.arange(nt))
    try:
        for eps, eps_loss, cap in CASES:
            r = ista(K, d, np.zeros(nt), cw=CW, lam=lam, eps=eps, eps_loss=eps_loss, cap=cap)
            ot, oit, odelta = O.proxgrad(exp, y, np.zeros(nt), cw=CW, lam=lam, epsilon=eps, epsilon_loss=eps_loss,
                                         max_iter=cap)
            what = (kind, eps, eps_loss, cap)
            assert r["iters"] == oit, (what, r["iters"], oit)
            assert close(r["theta"], ot), what
            assert np.array_equal(r["theta"] == 0.0, ot == 0.0), what
            if cap > 1:
                assert np.count_nonzero(r["theta"][d.m + 1:]) > 0, what
            x = ista(K, e, np.zeros(nt), cw=CW, lam=lam, eps=eps, eps_loss=eps_loss, cap=cap, entry="kmerlr_proxgrad")
            assert x["iters"] == r["iters"] and close(r["theta"], x["theta"]), what
    finally:
        e.free()


@pytest.mark.parametrize("kind", ["counts", "binarized", "f64", "subset"])
def test_fista_matches_the_restatement(K, oracle, c1, kind):
    """iteration counts, restarts, theta, y and t against accel_oracle.proxgrad_accel on the oracle's expansion"""
    O = oracle
    c = c1[kind]
    d, y, exp = c["d"], c["y"], c["exp"]
    nt = coeff_dim(d.m)
    lam = pair_lambda(O, c["ref"], y)
    restarts = 0
    for eps, eps_loss, cap in CASES:
        r = fista(K, d, np.zeros(nt), cw=CW, lam=lam, eps=eps, eps_loss=eps_loss, cap=cap)
        o = A.proxgrad_accel(exp, y, np.zeros(nt), cw=CW, lam=lam, epsilon=eps, epsilon_loss=eps_loss, max_iter=cap)
        what = (kind, eps, eps_loss, cap)
        assert r["iters"] == o["iters"] and r["restarts"] == o["restarts"], (what, r["iters"], o["iters"])
        assert close(r["theta"], o["theta"]) and close(r["y"], o["y"]), what
        assert np.array_equal(r["theta"] == 0.0, o["theta"] == 0.0), what
        assert r["t"] == o["t"], what
        restarts += r["restarts"]
    assert restarts > 0


# ---------------------------------------------------------------------------------------------------
# 4. the term list on both sides of PAIR_TERMS_MAX
# ---------------------------------------------------------------------------------------------------
def test_iterates_cross_pair_terms_max_both_ways(K, oracle, c1):
    """from theta = 0 at a small lambda the first step sets more than 8 192 pair coefficients (list -> O(q^2) walk);
    from a dense start at a large lambda it leaves fewer (walk -> list).  Both against the restatement."""
    O = oracle
    c = c1["counts"]
    d, y, exp = c["d"], c["y"], c["exp"]
    m, nt = d.m, coeff_dim(d.m)
    lam_up = pair_lambda(O, c["ref"], y, N=12000)
    rng = np.random.default_rng(4)
    lam_down = pair_lambda(O, c["ref"], y, N=200)
    # every coefficient non-zero, below the threshold s lambda: the first step zeroes all but the strong ones
    dense0 = np.concatenate([[0.1], rng.normal(scale=0.3 * step_pairs(d) * lam_down, size=nt - 1)])
    assert np.count_nonzero(dense0) == nt
    for start, lam, up in ((np.zeros(nt), lam_up, True), (dense0, lam_down, False)):
        one = ista(K, d, start, lam=lam, cap=1)
        k0, k1 = np.count_nonzero(start[m + 1:]), np.count_nonzero(one["theta"][m + 1:])
        assert (k0 <= 8192 < k1) if up else (k1 <= 8192 < k0), (k0, k1)
        r = ista(K, d, start, lam=lam, cap=12)
        ot, oit, _ = O.proxgrad(exp, y, start, lam=lam, epsilon=0.0, epsilon_loss=0.0, max_iter=12)
        assert r["iters"] == oit == 12 and close(r["theta"], ot, 1e-9 * np.max(np.abs(ot))), up
        a = fista(K, d, start, lam=lam, cap=12)
        o = A.proxgrad_accel(exp, y, start, lam=lam, epsilon=0.0, epsilon_loss=0.0, max_iter=12)
        bar = 1e-9 * np.max(np.abs(o["theta"]))
        assert a["restarts"] == o["restarts"] and close(a["theta"], o["theta"], bar) and close(a["y"], o["y"], bar), up


@pytest.fixture(scope="module")
def wide(K):
    """600 rows x 400 columns of small counts (79 800 pair coefficients, about 120 entries per row)"""
    rng = np.random.default_rng(6)
    n, m = 600, 400
    X = rng.integers(1, 4, size=(n, m)) * (rng.random((n, m)) < 0.3)
    rp = np.concatenate([[0], np.cumsum((X != 0).sum(1))]).astype(np.int64)
    d = K.from_csr(n, m, rp, np.nonzero(X)[1].astype(np.int32), X[X != 0].astype(np.float64))
    y = (rng.random(n) < 0.5).astype(np.uint8)
    d.SetLabels(y)
    yield d, y
    d.free()


@pytest.mark.parametrize("nterms", [0, 1, 8192, 8193, 50000])
def test_first_pass_is_the_gradient_of_kmerlr_gradient(K, wide, nterms):
    """at a theta with 0, 1, 8 192, 8 193 and 50 000 non-zero pair terms, lambda = 0: one step is theta - s g with g =
    kmerlr_gradient(cooccurrence = 1) bit for bit (the pass at theta uses its kernels and order), and the hook's loss
    after it is kmerlr_loss(theta', cooccurrence = 1, lambda = 0) within 2 ulp"""
    d, y = wide
    m, nt = d.m, coeff_dim(d.m)
    rng = np.random.default_rng(nterms + 1)
    theta = np.zeros(nt)
    theta[0] = -0.2
    theta[1:m + 1] = rng.normal(scale=1e-2, size=m)
    theta[m + 1 + rng.choice(nt - m - 1, nterms, replace=False)] = rng.normal(scale=1e-4, size=nterms)
    assert np.count_nonzero(theta[m + 1:]) == nterms
    g = K.logisticRegression(theta, CW, 0.0, Cooccurrence=True).Gradient(None, d)
    r = ista(K, d, theta, cw=CW, lam=0.0, eps_loss=1e-300, cap=1)
    assert r["iters"] == 1
    assert np.array_equal(r["theta"], theta - step_pairs(d) * g)
    lo = K.logisticRegression(r["theta"], CW, 0.0, Cooccurrence=True).Loss(d)
    assert abs(r["hook"][1] - lo) <= 2 * ULP * abs(lo)


# ---------------------------------------------------------------------------------------------------
# 5. m <= 44 and m = 1: the pair loop, never the reduced-matrix kernels
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("m", [1, 2, 30, 44])
def test_small_dim_runs_the_pair_loop(K, oracle, m):
    O = oracle
    rng = np.random.default_rng(m)
    n = 300
    X = rng.integers(0, 3, size=(n, m)) * (rng.random((n, m)) < 0.4)
    y = (rng.random(n) < 0.5).astype(np.uint8)
    X[y == 1, 0] += 1
    rp = np.concatenate([[0], np.cumsum((X != 0).sum(1))]).astype(np.int64)
    col, val = np.nonzero(X)[1].astype(np.int32), X[X != 0].astype(np.float64)
    d = K.from_csr(n, m, rp, col, val)
    d.SetLabels(y)
    nt = coeff_dim(m)
    assert nt <= 1024
    exp = O.reduce(O.from_csr(n, m, rp, col, val), np.arange(nt))
    e = K.select_data(d, np.arange(nt))
    try:
        lam = 1e-3
        launches = K.launch_count()
        r = ista(K, d, np.zeros(nt), cw=CW, lam=lam, eps_loss=1e-9, cap=2000)
        per = (K.launch_count() - launches) / (r["iters"] + 1)
        assert per > 3                      # one launch per batch would be the persistent reduced-matrix kernel
        ot, oit, _ = O.proxgrad(exp, y, np.zeros(nt), cw=CW, lam=lam, epsilon=0.0, epsilon_loss=1e-9, max_iter=2000)
        assert r["iters"] == oit and close(r["theta"], ot)
        x = ista(K, e, np.zeros(nt), cw=CW, lam=lam, eps_loss=1e-9, cap=2000, entry="kmerlr_proxgrad")
        assert x["iters"] == r["iters"] and close(x["theta"], r["theta"])
        # (300 steps: thousands of momentum steps without a restart amplify last-bit differences past the bar)
        a = fista(K, d, np.zeros(nt), cw=CW, lam=lam, eps_loss=1e-9, cap=300)
        o = A.proxgrad_accel(exp, y, np.zeros(nt), cw=CW, lam=lam, epsilon=0.0, epsilon_loss=1e-9, max_iter=300)
        assert a["iters"] == o["iters"] and a["restarts"] == o["restarts"] and close(a["theta"], o["theta"])
    finally:
        e.free()
        d.free()


# ---------------------------------------------------------------------------------------------------
# 6. slices and determinism
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("accel", [False, True])
def test_slices_and_determinism(K, oracle, c1, accel):
    """slices of 1 and 7 iterations (theta, y, t and hook_state carried) give one long call's bits; two runs likewise"""
    c = c1["counts"]
    d = c["d"]
    nt = coeff_dim(d.m)
    lam = pair_lambda(oracle, c["ref"], c["y"])
    run = (lambda **kw: fista(K, d, cw=CW, lam=lam, eps_loss=1e-9, **kw)) if accel else \
        (lambda **kw: ista(K, d, cw=CW, lam=lam, eps_loss=1e-9, **kw))
    a, b = run(theta=np.zeros(nt), cap=400), run(theta=np.zeros(nt), cap=400)
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    assert a["iters"] > 20
    for sl in (1, 7):
        st = dict(theta=np.zeros(nt), hook=np.array(NAN2))
        if accel:
            st.update(y=np.zeros(nt), t=1.0)
        done = 0
        while True:
            r = run(cap=min(sl, a["iters"] - done), **st)
            done += r["iters"]
            st = dict(theta=r["theta"], hook=r["hook"])
            if accel:
                st.update(y=r["y"], t=r["t"])
            if r["iters"] < sl or done >= a["iters"]:
                break
        assert done == a["iters"], sl
        for k in st:
            assert np.array_equal(st[k], a[k], equal_nan=True), (sl, k)


# ---------------------------------------------------------------------------------------------------
# 7. the estimator routes pair-mode fits of the whole space
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("accel", [False, True])
def test_estimator_routes_pair_space_fits(K, oracle, c1, accel):
    c = c1["counts"]
    d = c["d"]
    nt = coeff_dim(d.m)
    lam = pair_lambda(oracle, c["ref"], c["y"])
    est = K.KmerLrEstimator(Cooccurrence=True, EpsilonLoss=1e-9, MaxIterations=500, Accelerated=accel)
    est.ClassWeights = np.array(CW)
    est.Theta = np.zeros(nt)
    it, _ = est.estimate_proximal(d, lam)
    r = (fista if accel else ista)(K, d, np.zeros(nt), cw=CW, lam=lam, eps_loss=1e-9, cap=500)
    assert it == r["iters"] and np.array_equal(est.Theta, r["theta"])


# ---------------------------------------------------------------------------------------------------
# 8. launches per iteration
# ---------------------------------------------------------------------------------------------------
def test_launches_per_iteration_are_constant(K, wide):
    """the same launches per iteration with 0 and with all pair coefficients non-zero: ISTA 10 (flags, three scan
    launches, the list, rows, scatter_w, pairs_gradient, pass_tail, prox_update), FISTA one more"""
    d, _ = wide
    m, nt = d.m, coeff_dim(d.m)
    ista(K, d, np.zeros(nt), cap=1)                        # (the step size and the column view are built once)
    for accel, per in ((False, 10), (True, 11)):
        for start in (np.zeros(nt), np.full(nt, 1e-6)):
            counts = []
            for cap in (16, 32):
                l0 = K.launch_count()
                r = (fista if accel else ista)(K, d, start, lam=0.0, cap=cap)
                assert r["iters"] == cap
                counts.append(K.launch_count() - l0)
            assert counts[1] - counts[0] == 16 * per, (accel, counts)


# ---------------------------------------------------------------------------------------------------
# 9. refusals
# ---------------------------------------------------------------------------------------------------
def test_refusals(K, c1):
    """KMERLR_ERR_ARG with a message: ntheta other than kmerlr_coeff_dim(m), a null theta, y, t or class_w, t < 1 or not
    finite, a matrix without labels, an empty set.  (A sharded matrix is refused too; that needs more than one rank and
    is not exercised here.)"""
    from kmerlr_b200 import _lib
    L = _lib.lib()
    d = c1["counts"]["d"]
    nt = coeff_dim(d.m)
    nolab = K.from_dense(np.eye(4))
    empty = K.from_dense(np.zeros((0, 5)))
    empty.SetLabels(np.zeros(0, dtype=np.uint8))

    def refused(match, f, *a, **kw):
        with pytest.raises(K.KmerLrError) as e:
            f(*a, **kw)
        assert e.value.code == _lib.ERR_ARG and match in str(e.value), str(e.value)

    try:
        for f in (ista, fista):
            refused("kmerlr_coeff_dim", f, K, d, np.zeros(d.m + 1), cap=3)
            refused("kmerlr_coeff_dim", f, K, d, np.zeros(nt + 1), cap=3)
            refused("no labels", f, K, nolab, np.zeros(coeff_dim(4)), cap=3)
            refused("empty", f, K, empty, np.zeros(coeff_dim(5)), cap=3)
        for t in (0.5, 0.0, -1.0, float("nan"), float("inf")):
            refused("momentum t", fista, K, d, np.zeros(nt), t=t, cap=3)
        th, y, cw = np.zeros(nt), np.zeros(nt), np.ones(2)
        hk, it, de, rs, t = np.array(NAN2), C.c_int64(), C.c_double(), C.c_int64(), C.c_double(1.0)
        for args in ((None, _p(y), t, _p(cw)), (_p(th), None, t, _p(cw)), (_p(th), _p(y), None, _p(cw)),
                     (_p(th), _p(y), t, None)):
            refused("null argument", lambda: _lib.check(L.kmerlr_proxgrad_pairs_accel(
                d.h, args[0], args[1], args[2], nt, args[3], 1e-3, 0.0, 1.0, 0.0, 0.0, 3, _p(hk), it, de, rs)))
        for args in ((None, _p(cw)), (_p(th), None)):
            refused("null argument", lambda: _lib.check(L.kmerlr_proxgrad_pairs(
                d.h, args[0], nt, args[1], 1e-3, 0.0, 1.0, 0.0, 0.0, 3, _p(hk), it, de)))
        s = C.c_double()
        refused("empty", lambda: _lib.check(L.kmerlr_step_size_pairs(empty.h, 0.0, 1.0, s)))
    finally:
        nolab.free()
        empty.free()


# ---------------------------------------------------------------------------------------------------
# 10. C4 scale
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def c4(K):
    """the 16 000 training rows of fold 0 of C4 (k = 1..6 revcomp, m = 2 772, 3 843 379 coefficients), u32 counts"""
    from kmerlr_b200 import synth
    buf, off, y = synth.training_set(10000, 10000, 500)
    n = len(off) - 1
    tr = np.nonzero(np.arange(n) % 5 != 0)[0]
    lens = np.diff(off)
    o = np.concatenate([[0], np.cumsum(lens[tr])]).astype(np.int64)
    b = np.concatenate([buf[off[i]:off[i + 1]] for i in tr])
    d = K.compile_test_data(None, K.NewKmerCounter(1, 6, revcomp=True), None, None, True, False, (b, o))
    yt = y[tr].astype(np.uint8)
    d.SetLabels(yt)
    assert d.n == 16000 and d.m == 2772 and coeff_dim(d.m) == 3843379
    yield d, yt
    d.free()


def torch_model(torch, X, theta, iu):
    """z of the pair-mode predictor in fp64 on the device: theta_0 + X theta_s + 1/2 rowsum((X Theta) * X), Theta the
    symmetric matrix of the pair coefficients"""
    m = X.shape[1]
    T = torch.zeros((m, m), dtype=torch.float64, device=X.device)
    T[iu[0], iu[1]] = theta[m + 1:]
    T = T + T.T
    return theta[0] + X @ theta[1:m + 1] + 0.5 * ((X @ T) * X).sum(1)


def torch_grad(torch, X, yl, theta, iu, cw):
    """the gradient of the mean weighted log-loss: bias, X^T w, and the upper triangle of X^T diag(w) X"""
    z = torch_model(torch, X, theta, iu)
    x = -z
    r = -torch.where(x > 0.0, x + torch.log1p(torch.exp(-x.abs())), torch.log1p(torch.exp(torch.clamp(x, max=0.0))))
    n = X.shape[0]
    w = torch.where(yl == 1, cw[1] / n * (torch.exp(r) - 1.0), cw[0] / n * torch.exp(r))
    P = X.T @ (w[:, None] * X)
    return torch.cat([w.sum()[None], X.T @ w, P[iu[0], iu[1]]])


def torch_fista(torch, X, yl, theta, iu, cw, lam, s, iters):
    """accel_oracle.proxgrad_accel (no hook, no stopping rule) in torch fp64"""
    th, y, t, restarts = theta.clone(), theta.clone(), 1.0, 0
    for _ in range(iters):
        tn = y - s * torch_grad(torch, X, yl, y, iu, cw)
        tn[1:] = torch.sign(tn[1:]) * torch.clamp(tn[1:].abs() - s * lam, min=0.0)
        dl = tn - th
        if float(torch.dot(y - tn, dl)) > 0.0:
            t, y, restarts = 1.0, tn.clone(), restarts + 1
        else:
            t1 = (1.0 + (1.0 + 4.0 * t * t) ** 0.5) / 2.0
            y, t = tn + ((t - 1.0) / t1) * dl, t1
        th = tn
    return th, y, t, restarts


def test_c4_fista_against_dense_restatement_and_kkt(K, c4):
    """30 FISTA iterations at the lambda of the first Select at N = 20 over the pair space against a dense fp64
    restatement on the device (theta and y within 1e-9 of max |theta|); then a fit warm-started from the leapfrog
    epoch's model, capped at 400 iterations: the KKT conditions hold within 20 % of lambda at its theta (0.16 lambda after
    150 iterations on one NVIDIA B200) and its F is at most the leapfrog model's F embedded in the pair space"""
    torch = pytest.importorskip("torch")
    d, yl = c4
    m, nt = d.m, coeff_dim(d.m)
    cw = (1.0, 1.0)
    est = K.KmerLrEstimator(Cooccurrence=True, EpsilonLoss=1e-8, MaxEpochs=1, Accelerated=True, tie=K.TIE_INDEX)
    est.estimate_loop(d, 20)
    lam = est.path[0][0]
    assert lam > 0.0
    warm = np.zeros(nt)
    warm[0] = est.Theta[0]
    warm[est.active_idx] = est.Theta[1:]
    s = step_pairs(d)
    r = fista(K, d, np.zeros(nt), cw=cw, lam=lam, cap=30)
    assert r["iters"] == 30
    rp, col, val = rows_of(d)
    X = torch.zeros((d.n, m), dtype=torch.float64, device="cuda")
    X[torch.repeat_interleave(torch.arange(d.n, device="cuda"), torch.as_tensor(np.diff(rp), device="cuda")),
      torch.as_tensor(col.astype(np.int64), device="cuda")] = torch.as_tensor(val, device="cuda")
    iu = torch.triu_indices(m, m, 1, device="cuda")
    yt = torch.as_tensor(yl, device="cuda")
    th, y, t, restarts = torch_fista(torch, X, yt, torch.zeros(nt, dtype=torch.float64, device="cuda"), iu, cw, lam, s, 30)
    scale = float(th.abs().max())
    assert np.count_nonzero(r["theta"][m + 1:]) > 0
    assert np.max(np.abs(r["theta"] - th.cpu().numpy())) <= 1e-9 * scale
    assert np.max(np.abs(r["y"] - y.cpu().numpy())) <= 1e-9 * scale
    assert r["restarts"] == restarts and abs(r["t"] - t) <= 1e-12 * t
    del X, th, y
    torch.cuda.empty_cache()

    def F(theta):
        return K.logisticRegression(theta, cw, 0.0, Cooccurrence=True).Loss(d) + lam * np.sum(np.abs(theta[1:]))

    f = fista(K, d, warm, cw=cw, lam=lam, eps_loss=1e-12, cap=400)
    g = K.logisticRegression(f["theta"], cw, 0.0, Cooccurrence=True).Gradient(None, d)
    th = f["theta"]
    nz = th[1:] != 0.0
    res = np.where(nz, np.abs(g[1:] + lam * np.sign(th[1:])), np.maximum(np.abs(g[1:]) - lam, 0.0))
    print("C4: lambda %.6g, %d iterations, %d restarts, %d non-zero, KKT residual %.3g lambda, F %.12g vs leapfrog %.12g"
          % (lam, f["iters"], f["restarts"], int(nz.sum()), res.max() / lam, F(th), F(warm)))
    assert abs(g[0]) <= 0.2 * lam
    assert res.max() <= 0.2 * lam
    assert F(th) <= F(warm)
