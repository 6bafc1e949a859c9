"""The reduced-matrix solver (proxgrad on <= 1023 columns: fused_small_kernel, fused_small_persistent on the rows, on the
sliced + column-major views and on the block-local view) and the coordinate estimator at the shapes, magnitudes and
tunables where their fixed-point sums can break.  Needs a B200.

Both accumulate in 64-bit fixed point.  The reduced solver uses the scales of the full-space pass (DESIGN section 4.2):
e = 60 - ceil(log2(max|cw| max|v|)) for the columns, 60 - ceil(log2(max|cw| max(max|v|, 1))) for the bias, so one of
its iterations from theta = (b, 0, ..., 0) is a host prox step on fused_kernel's gradient bit for bit.  The coordinate
estimator gives the Gram entries and xy of the bias and of the columns their own exponents (DESIGN section 4.3b), so a
matrix scaled by a power of two gives the same integers."""
import ctypes as C
import math

import numpy as np
import pytest
import scipy.sparse as sp

from test_gradient_edges_gpu import EPS, LD, check_against, csr_case, reference

pytestmark = pytest.mark.gpu

DEFAULTS = {"small_long": -1, "persistent": 1, "persist_bps": 0}
# every order-only tunable of the reduced solver: the row pass, the sliced + column-major views, the block-local view;
# the cooperative persistent kernel or one launch per iteration; the resident blocks per SM of the persistent grid
TUNABLES = [(sl, pe, bps) for sl in (-1, 0, 1, 2) for pe in (0, 1) for bps in (0, 1, 2)]


def restore(K):
    for k, v in DEFAULTS.items():
        K.option(k, v)


def set_tunables(K, t):
    K.option("small_long", t[0])
    K.option("persistent", t[1])
    K.option("persist_bps", t[2])


def sm_count():
    try:
        import torch
        return torch.cuda.get_device_properties(0).multi_processor_count
    except Exception:                                      # (the card the grid sizes below were chosen for)
        return 148


# n = 64 * (blocks of one wave) +- 1: one row past / short of 64 rows in every block of the first wave
WAVE = 64 * sm_count() * 6


def step_size(K, d):
    from kmerlr_b200 import _lib
    out = C.c_double()
    _lib.check(_lib.lib().kmerlr_step_size(d.h, 0.0, 1.0, out))
    return out.value


def matrix(rng, n, m, lens, kind):
    """csr_case, plus the kinds scaled by a power of two ("p20", "p40": negreal times 2^-20, 2^-40; theta times 2^k)"""
    if kind in ("p20", "p40"):
        k = int(kind[1:])
        rowptr, col, val, theta = csr_case(rng, n, m, lens, "negreal")
        theta[1:] = np.ldexp(theta[1:], k)
        return rowptr, col, np.ldexp(val, -k), theta
    return csr_case(rng, n, m, lens, kind)


def labels(rng, n):
    y = (rng.random(n) < 0.4).astype(np.uint8)
    if n > 1:
        y[0], y[1] = 1, 0
    return y


def prox(theta, g, step, lam):
    """the prox step of small_tail / prox_update in float64 (the library builds with --fmad=false)"""
    t = theta - step * g
    thr = step * lam
    a = np.maximum(np.abs(t[1:]) - thr, 0.0)
    t[1:] = np.where(t[1:] >= 0.0, a, -a)
    return t


def run(K, d, theta, cw, lam, cap, eps=0.0, eps_loss=0.0):
    est = K.KmerLrEstimator(Epsilon=eps, EpsilonLoss=eps_loss, MaxIterations=cap)
    est.Theta, est.ClassWeights = np.array(theta, dtype=np.float64), np.array(cw, dtype=np.float64)
    it, delta = est.estimate_proximal(d, lam)
    return est.Theta, it, delta, est.hook_state.copy()


SHORT, MID, LONG = (0, 1, 4, 7), (4, 7, 8), (0, 1, 4, 7, 8, 31, 32, 33, 1023)   # < 4, 4..8, > 8 entries per row
CASES = [  # n, m, row lengths (capped at m), values, class weights, lambda as a share of the median |g_j|
    (1, 1, (1,), "counts", (1.0, 1.0), 0.0),
    (31, 2, SHORT, "tiny", (0.7, 1.9), 0.5),
    (33, 31, MID, "p20", (1e-3, 1e3), 0.0),
    (WAVE - 1, 32, LONG, "p40", (1.0, 1.0), 0.5),
    (WAVE + 1, 33, LONG, "negreal", (0.7, 1.9), 0.5),
    (70001, 1023, MID, "counts", (1e-3, 1e3), 0.5),
    (70001, 33, LONG, "mixed", (1.0, 1.0), 0.0),
    (31, 1023, LONG, "p20", (0.7, 1.9), 0.0),
    (WAVE + 1, 1023, SHORT, "tiny", (1.0, 1.0), 0.5),
    (33, 1023, SHORT, "counts", (1.0, 1.0), 0.5),
    (WAVE - 1, 2, MID, "mixed", (1e-3, 1e3), 0.5),
    (1, 33, (33,), "negreal", (0.7, 1.9), 0.0),
    (70001, 31, LONG, "p40", (1e-3, 1e3), 0.0),
    (31, 32, LONG, "tiny", (1e-3, 1e3), 0.5),
    (33, 1, SHORT, "p20", (1.0, 1.0), 0.5),
]
IDS = ["n%d-m%d-%s-%s-cw%g" % (c[0], c[1], "x".join(map(str, c[2])), c[3], c[4][1]) for c in CASES]


# ---------------------------------------------------------------------------------------------------
# (a) one reduced iteration from theta = (b, 0, ..., 0) is one host prox step on fused_kernel's gradient
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,m,lens,kind,cw,lamf", CASES, ids=IDS)
def test_one_reduced_iteration_is_a_prox_step_on_the_full_gradient(K, n, m, lens, kind, cw, lamf):
    """z_i = b exactly on both paths, so the weights have the same bits; the reduced kernels must then add the same
    integers as fused_kernel, and small_tail must take the same prox step, under every order-only tunable"""
    rng = np.random.default_rng(n * 11 + m)
    rowptr, col, val, _ = matrix(rng, n, m, lens, kind)
    y = labels(rng, n)
    d = K.from_csr(n, m, rowptr, col if len(col) else [0], val if len(val) else [0.0])
    try:
        d.SetLabels(y)
        theta = np.zeros(m + 1)
        theta[0] = -0.4
        g = K.logisticRegression(theta, cw).Gradient(None, d)
        lam = lamf * float(np.median(np.abs(g[1:])))
        want = prox(theta, g, step_size(K, d), lam)
        assert np.count_nonzero(want[1:]) > 0
        for t in TUNABLES:
            set_tunables(K, t)
            th, it, _, _ = run(K, d, theta, cw, lam, 1)
            assert it == 1, t
            bad = np.nonzero(th != want)[0]
            assert len(bad) == 0, "%s: %d of %d coefficients differ, first j=%d: %r vs %r" % (
                t, len(bad), m + 1, bad[0], th[bad[0]], want[bad[0]])
    finally:
        restore(K)
        d.free()


# ---------------------------------------------------------------------------------------------------
# (b) one iteration from a general theta against long double
# ---------------------------------------------------------------------------------------------------
def check_step(ref, theta, th, step, lam, what):
    """theta_1 against the long-double prox step on the reference gradient: step * gb_j, plus one rounding each
    for the product, the difference, the threshold and the shrunk value"""
    t = LD(1) * theta - LD(step) * ref["g"]
    a = np.maximum(np.abs(t[1:]) - LD(step) * LD(lam), LD(0))
    t[1:] = np.where(t[1:] >= 0, a, -a)
    p = np.abs(step * ref["g"].astype(np.float64))
    # the roundings of step * g, theta - step * g (at most |theta| + p), step * lambda and |t| - step * lambda
    bound = step * ref["gb"] + 2.0 * EPS * (2.0 * p + np.abs(theta) + step * lam + np.abs(th)) + 1e-300
    err = np.abs((th.astype(LD) - t).astype(np.float64))
    bad = np.nonzero(err > bound)[0]
    assert len(bad) == 0, "%s: %d of %d coefficients off, worst j=%d err=%.3e bound=%.3e (e=%d, e0=%d)" % (
        what, len(bad), len(th), bad[np.argmax(err[bad] / bound[bad])], np.max(err[bad]), bound[bad[0]], ref["e"],
        ref["e0"])


def dense_transformed(K, rng, n, m):
    """Transform.Apply with an offset: dense rows with negative values and every column present"""
    rowptr, col, val, _ = csr_case(rng, n, m, (1, 4, 7), "counts")
    d = K.from_csr(n, m, rowptr, col, val)
    off = np.concatenate([[0.0], rng.uniform(0.5, 2.5, m)])
    sc = np.concatenate([[1.0], rng.uniform(1e-3, 0.3, m)])
    td = K.Transform(Offset=off, Scale=sc).Apply(d)
    d.free()
    return td


B_CASES = CASES + [(5000, 40, None, "transformed", (0.7, 1.9), 0.5), (2000, 1023, None, "transformed", (1.0, 1.0), 0.0)]
B_IDS = IDS + ["n%d-m%d-transformed" % (c[0], c[1]) for c in B_CASES[len(CASES):]]


@pytest.mark.parametrize("n,m,lens,kind,cw,lamf", B_CASES, ids=B_IDS)
def test_one_reduced_iteration_against_long_double(K, n, m, lens, kind, cw, lamf):
    rng = np.random.default_rng(n * 13 + m)
    if kind == "transformed":
        d = dense_transformed(K, rng, n, m)
        rowptr, col, val = d.rows()
        assert np.min(val) < 0.0 and len(val) == n * m
        theta = rng.normal(scale=1.0 / (0.3 * math.sqrt(m + 1.0)), size=m + 1)
    else:
        rowptr, col, val, theta = matrix(rng, n, m, lens, kind)
        d = K.from_csr(n, m, rowptr, col if len(col) else [0], val if len(val) else [0.0])
    y = labels(rng, n)
    try:
        d.SetLabels(y)
        ref = reference(n, m, rowptr, col, val, y, theta, cw, serial=True)
        lam = lamf * float(np.median(np.abs(ref["g"][1:].astype(np.float64))))
        step = step_size(K, d)
        for t in ((-1, 1, 0), (0, 0, 0), (1, 1, 0)):
            set_tunables(K, t)
            th, it, _, _ = run(K, d, theta, cw, lam, 1)
            assert it == 1, t
            check_step(ref, theta, th, step, lam, "%s %s" % (kind, t))
    finally:
        restore(K)
        d.free()


# ---------------------------------------------------------------------------------------------------
# (c) order-only tunables over many iterations
# ---------------------------------------------------------------------------------------------------
def edge_matrix(rng, n, m, lens, vmax):
    """integer values 1..5 with vmax and vmax - 1 among them; the first, the last and a middle column empty"""
    inner = m - 3
    rowptr, col, val, _ = csr_case(rng, n, inner, lens, "counts")
    col = (col + 1 + (col >= inner // 2)).astype(np.int32)
    if len(val):
        at = rng.choice(len(val), size=min(len(val), 5), replace=False)
        val[at[0]] = vmax
        val[at[1:]] = vmax - 1
    return rowptr, col, val


def pack_limit(n):
    """ensure_packed: counts below 2^min(32 - rb, 22), rb = the bits of a row index"""
    rb = max(1, math.ceil(math.log2(n)))
    return 2 ** min(32 - rb, 22)


def blockview_limit(n):
    """ensure_blockview for n <= 64 * (SMs): one block per 64 rows, counts below 2^(22 - bits of a block's rows)"""
    g = (n + 63) // 64
    rows = (n + g - 1) // g + 1
    return 2 ** (22 - max(1, math.ceil(math.log2(rows))))


ORDER_CASES = [  # n, m, row lengths, largest value
    (4096, 40, (0, 1, 4, 7, 8, 31, 32, 33), pack_limit(4096) - 1),      # packs, too large for the block-local view
    (4097, 40, (0, 1, 4, 7, 8, 31, 32, 33), pack_limit(4097)),          # does not pack: rb went up with n
    (4096, 40, (0, 4, 7, 8, 12), blockview_limit(4096) - 1),            # every view
    (4097, 40, (0, 4, 7, 8, 12), blockview_limit(4097)),                # packs, the block-local view refuses
    (4097, 1023, (0, 1, 4, 7, 8, 31, 32, 33, 1023), 5),
    (1000, 6, (0,), 1),                                                 # nnz = 0
]


@pytest.mark.parametrize("n,m,lens,vmax", ORDER_CASES, ids=["n%d-m%d-v%d" % (c[0], c[1], c[3]) for c in ORDER_CASES])
def test_order_only_tunables_are_bit_identical(K, n, m, lens, vmax):
    assert sm_count() * 64 >= n                            # (blockview_limit's grid: one block per 64 rows)
    rng = np.random.default_rng(n + m + vmax)
    rowptr, col, val = edge_matrix(rng, n, m, lens, vmax)
    y = labels(rng, n)
    d = K.from_csr(n, m, rowptr, col if len(col) else [0], val if len(val) else [0.0])
    try:
        assert d.nnz == len(val)
        if len(val):
            counts = np.bincount(col, minlength=m)
            assert counts[0] == 0 and counts[-1] == 0 and counts[(m - 3) // 2 + 1] == 0 and np.max(val) == vmax
        d.SetLabels(y)
        cw = (0.8, 1.3)
        # the loss-based stop: twice the loss decrement of the 60th iteration stops the run at the 60th at the latest,
        # whatever the matrix (a fixed threshold can sit below every decrement of a slowly converging problem)
        restore(K)
        hook = run(K, d, np.zeros(m + 1), cw, 1e-4, 60, eps_loss=1e-300)[3]
        stop_loss = max(2.0 * abs(hook[0] - hook[1]), 1e-300)
        assert np.isfinite(stop_loss)
        for cap, eps_loss in ((60, 0.0), (100000, stop_loss), (0, 0.0)):
            first = None
            for t in TUNABLES:
                set_tunables(K, t)
                r = run(K, d, np.zeros(m + 1), cw, 1e-4, cap, eps_loss=eps_loss)
                if cap == 60:
                    assert r[1] == 60 or len(val) == 0, (t, r[1])
                if cap == 100000:
                    assert r[1] <= 60, (t, r[1])
                if first is None:
                    first = (t, r)
                    continue
                what = (t, first[0], cap)
                assert np.array_equal(r[0], first[1][0]), what
                assert r[1] == first[1][1], what
                assert r[2] == first[1][2] or (np.isnan(r[2]) and np.isnan(first[1][2])), what
                assert np.array_equal(r[3], first[1][3], equal_nan=True), what
    finally:
        restore(K)
        d.free()


# ---------------------------------------------------------------------------------------------------
# (d) coordinate estimator: power-of-two invariance
# ---------------------------------------------------------------------------------------------------
def coordinate(K, d, theta, cap, l1=0.0, l2=0.0, eps=0.0, eps_loss=0.0, cwh=(1.0, 1.0)):
    est = K.KmerLrEstimator(Epsilon=eps, EpsilonLoss=eps_loss, L2Reg=l2, MaxIterations=cap)
    est.Theta, est.ClassWeights, est.L1Reg = np.array(theta, dtype=np.float64), np.array(cwh), l1
    sweeps, delta = est.estimate_coordinate(d)
    return est.Theta, sweeps, delta


def dense(rng, n, m, vmax):
    """dense rows, values uniform in +-vmax (one of them vmax itself)"""
    X = rng.uniform(-vmax, vmax, (n, m))
    X[0, 0] = vmax
    rowptr = np.arange(n + 1, dtype=np.int64) * m
    col = np.tile(np.arange(m, dtype=np.int32), n)
    return rowptr, col, X.ravel()


@pytest.mark.parametrize("k", [1, 12, 30])
def test_coordinate_power_of_two_invariance(K, k):
    """X' = 2^-k X, theta' = (theta_0, 2^k theta): the same z and weights, and with exponents that follow max|v| the
    same Gram and xy integers, so theta'_out = (theta_0_out, 2^k theta_out) bit for bit after the same sweeps"""
    rng = np.random.default_rng(7)
    n, m = 1200, 20
    rowptr, col, val = dense(rng, n, m, 0.5)
    y = (rng.random(n) < 0.3).astype(np.uint8)
    theta = rng.normal(scale=0.1, size=m + 1)
    ts = theta.copy()
    ts[1:] = np.ldexp(theta[1:], k)
    d, ds = K.from_csr(n, m, rowptr, col, val), K.from_csr(n, m, rowptr, col, np.ldexp(val, -k))
    try:
        d.SetLabels(y); ds.SetLabels(y)
        th, sw, _ = coordinate(K, d, theta, 12)
        ths, sws, _ = coordinate(K, ds, ts, 12)
        assert np.all(np.isfinite(th)) and np.all(np.isfinite(ths)), "scaled by 2^-%d: not finite" % k
        assert sws == sw
        assert ths[0] == th[0]
        assert np.array_equal(ths[1:], np.ldexp(th[1:], k)), "%d of %d columns differ" % (
            int(np.sum(ths[1:] != np.ldexp(th[1:], k))), m)
    finally:
        d.free(); ds.free()


# ---------------------------------------------------------------------------------------------------
# (e) coordinate estimator at small magnitudes and at its size limit, against the numpy restatement
# ---------------------------------------------------------------------------------------------------
# the grid of test_coordinate_estimator_matches_restatement; L1 and L2 in units of max|v| and max|v|^2 (xy and the
# Gram diagonal scale with them)
CD_GRID = [(0.0, 0.0, 0.0, 0.0, 25), (1e-4, 0.0, 2.0, 0.0, 5000), (1e-3, 0.0, 20.0, 0.5, 5000), (0.0, 1e-6, 1.0, 0.0, 5000),
           (0.0, 0.0, 1.0, 0.0, 0)]


def coordinate_vs_oracle(K, O, n, m, rowptr, col, val, y, grid, vmax):
    d = K.from_csr(n, m, rowptr, col, val)
    om = O.from_csr(n, m, rowptr, col, val)
    cwh = np.array([0.9, 1.2])
    try:
        d.SetLabels(y)
        for eps, eps_loss, l1, l2, cap in grid:
            l1, l2 = l1 * vmax, l2 * vmax * vmax
            th, sw, delta = coordinate(K, d, np.zeros(m + 1), cap, l1, l2, eps, eps_loss, cwh)
            oth, osw, odelta = O.coordinate(om, y, np.zeros(m + 1), cwh, l1, l2, eps, eps_loss, cap)
            what = (vmax, m, eps, eps_loss, l1, cap)
            assert np.all(np.isfinite(oth)), what
            assert sw == osw, (what, sw, osw)
            err = np.max(np.abs(th - oth))
            assert err <= 1e-8 * np.max(np.abs(oth)), (what, err, np.max(np.abs(oth)))
            assert np.array_equal(th == 0.0, oth == 0.0), what
    finally:
        d.free()


@pytest.mark.parametrize("vmax", [1e-3, 1e-6, 1e-8])
def test_coordinate_small_values_against_restatement(K, oracle, vmax):
    """one positive row in 2 000: an IRLS class weight of 1 000"""
    rng = np.random.default_rng(8)
    n, m = 2000, 25
    rowptr, col, val, _ = csr_case(rng, n, m, (3, 8, 12, 25), "negreal")
    val = val * (vmax / np.max(np.abs(val)))
    y = np.zeros(n, dtype=np.uint8)
    y[777] = 1
    coordinate_vs_oracle(K, oracle, n, m, rowptr, col, val, y, CD_GRID, vmax)


@pytest.mark.parametrize("m,vmax", [(31, 1e-3), (32, 1.0), (33, 1e-6), (1023, 1e-3)])
def test_coordinate_dense_rows_at_the_size_limit(K, oracle, m, vmax):
    """m = 1023: ntheta = 1024, every thread of cd_sweep_kernel live; (m + 1)^2 atomics per row in the row pass"""
    rng = np.random.default_rng(9 + m)
    n = 1500
    rowptr, col, val = dense(rng, n, m, vmax)
    y = (rng.random(n) < 0.3).astype(np.uint8)
    grid = [(0.0, 0.0, 0.0, 1.0, 4)] if m == 1023 else CD_GRID[:3]
    coordinate_vs_oracle(K, oracle, n, m, rowptr, col, val, y, grid, vmax)


def test_coordinate_refuses_1024_columns(K):
    rng = np.random.default_rng(10)
    n, m = 50, 1024
    rowptr, col, val = dense(rng, n, m, 1.0)
    d = K.from_csr(n, m, rowptr, col, val)
    try:
        d.SetLabels((np.arange(n) % 2).astype(np.uint8))
        with pytest.raises(K.KmerLrError):
            coordinate(K, d, np.zeros(m + 1), 3)
    finally:
        d.free()


# ---------------------------------------------------------------------------------------------------
# (f) the reduced solver over many iterations on small values, against the oracle
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [20, 40])
def test_reduced_solver_small_values_against_oracle(K, oracle, k):
    """every column against its own magnitude: the bias dominates max|theta| when the features are this small"""
    O = oracle
    rng = np.random.default_rng(11 + k)
    n, m = 3000, 60
    rowptr, col, val, _ = csr_case(rng, n, m, (0, 1, 4, 7, 8, 31), "negreal")
    val = np.ldexp(val, -k)
    y = labels(rng, n)
    cw = (0.7, 1.9)
    d = K.from_csr(n, m, rowptr, col, val)
    om = O.from_csr(n, m, rowptr, col, val)
    try:
        d.SetLabels(y)
        assert step_size(K, d) == O.step_size(om)
        for lam, eps_loss, cap in ((0.0, 0.0, 60), (2.0 ** -k * 1e-4, 1e-10, 100000)):
            oth, oit, _ = O.proxgrad(om, y, np.zeros(m + 1), cw, lam, epsilon=0.0, epsilon_loss=eps_loss, max_iter=cap)
            if cap == 60:
                assert oit == 60
            else:
                assert 1 < oit < cap
            th, it, _, _ = run(K, d, np.zeros(m + 1), cw, lam, cap, eps_loss=eps_loss)
            assert it == oit, (lam, it, oit)
            err = np.abs(th - oth)
            bound = 1e-9 * np.abs(oth)
            bound[1:] += 1e-12 * np.max(np.abs(oth[1:]))
            bound[0] += 1e-12 * abs(oth[0])
            bad = np.nonzero(err > bound)[0]
            assert len(bad) == 0, "2^-%d, lambda %g: %d of %d coefficients off, worst j=%d: %r vs %r" % (
                k, lam, len(bad), m + 1, bad[np.argmax(err[bad] / bound[bad])], th[bad[0]], oth[bad[0]])
            assert np.array_equal(th == 0.0, oth == 0.0)
    finally:
        d.free()
