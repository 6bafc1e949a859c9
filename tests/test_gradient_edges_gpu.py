"""The fixed-point gradient, the fused pass tail and the device top-2N select at the sizes, magnitudes and tunables
where they can break.  Needs a B200.

The gradient is accumulated in 64-bit fixed point: a column sum is exact up to one rounding of 2^-e per stored entry
(CSR pass) or per position (matrix-free pass), e = 60 - ceil(log2(max|cw| max|v|)) for the columns and
60 - ceil(log2(max|cw| max(max|v|, 1))) for the bias (DESIGN section 4.2).  Every column is checked against a
long-double reference with that bound plus the fp64 error of the weight, z and the product; a relative tolerance on
max |g| would let an error confined to the small columns through."""
import math

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

if np.finfo(np.longdouble).nmant < 63:
    pytest.skip("the reference needs an extended long double (64-bit mantissa or more)", allow_module_level=True)

EPS = 2.0 ** -53
LD = np.longdouble
DEFAULTS = {"hot_cols": 6144, "fused_ticket": 8, "implicit": 1, "super_len": -1}


def restore(K):
    for k, v in DEFAULTS.items():
        K.option(k, v)


# ---------------------------------------------------------------------------------------------------
# reference and per-column precision contract
# ---------------------------------------------------------------------------------------------------
def scale_exponents(val, cw):
    """(columns, bias): the exponents of the fixed-point scales"""
    vmax = float(np.max(np.abs(val))) if len(val) else 0.0
    cmax = max(abs(cw[0]), abs(cw[1]))

    def ex(bound):
        return min(60 - math.ceil(math.log2(bound)), 1000)
    return ex(cmax * (vmax if vmax > 0.0 else 1.0)), ex(cmax * max(vmax, 1.0))


def reference(n, m, rowptr, col, val, y, theta, cw, serial=False):
    """z = X theta, the weights w_i and g_j = sum_i w_i v_ij in long double, with the allowed error of every z_i,
    g_j and of the loss.  serial: z sums a row in entry order (the reduced-matrix kernels), not in 32-lane strides"""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    col = np.asarray(col, dtype=np.int32)
    val = np.asarray(val, dtype=np.float64)
    lab = np.asarray(y).astype(bool)
    th = np.asarray(theta, dtype=np.float64)
    X = sp.csr_matrix((val.astype(LD), col, rowptr), shape=(n, m))
    z = LD(th[0]) + X @ th[1:].astype(LD)
    A = sp.csr_matrix((np.abs(val), col, rowptr), shape=(n, m))
    Z = abs(th[0]) + A @ np.abs(th[1:])                   # |theta_0| + sum_k |v_ik theta_k|
    q = np.diff(rowptr)
    # z on the device: per-lane partial sums of 32-strided entries, a shuffle tree, theta_0, the products; or one
    # serial sum of q products plus theta_0
    kz = q + 2.0 if serial else np.maximum(8, np.ceil(q / 32.0) + 7)
    cw0, cw1, cmax = LD(cw[0]), LD(cw[1]), max(abs(cw[0]), abs(cw[1]))
    w = np.where(lab, -cw1 / (1 + np.exp(z)), cw0 / (1 + np.exp(-z))) / LD(n)
    term = np.where(lab, cw1 * np.logaddexp(LD(0), -z), cw0 * np.logaddexp(LD(0), z))
    g = np.empty(m + 1, dtype=LD)
    g[0] = w.sum()
    g[1:] = X.T @ w
    wf = np.abs(w.astype(np.float64))
    # the fp64 weight: its own rounding, the z error through dw/dz <= cw / (4 n), exp(r) - 1 near 1
    dw = EPS * (8.0 * wf + cmax / n * (2.0 + kz * Z / 4.0))
    e, e0 = scale_exponents(val, cw)
    gb = np.empty(m + 1)
    gb[0] = 2.0 ** -e0 * (0.5 * n + 1.0) + dw.sum()
    per = np.bincount(col, weights=np.maximum(1.0, np.abs(val)), minlength=m) if len(col) else np.zeros(m)
    gb[1:] = 2.0 ** -e * (0.5 * per + 1.0) + A.T @ dw
    tf = np.abs(term.astype(np.float64))
    loss_bound = 64.0 * EPS * tf.sum() / n + float(np.sum(wf * kz * EPS * Z)) + EPS * float(abs(term.sum() / n))
    return dict(z=z, zb=kz * EPS * Z, g=g, gb=gb, loss=term.sum() / LD(n), lb=loss_bound, e=e, e0=e0)


def check_against(ref, g=None, z=None, loss=None, what=""):
    if g is not None:
        err = np.abs((np.asarray(g, dtype=LD) - ref["g"]).astype(np.float64))
        bad = np.nonzero(err > ref["gb"])[0]
        assert len(bad) == 0, "%s: %d columns off, worst j=%d err=%.3e bound=%.3e (e=%d)" % (
            what, len(bad), bad[np.argmax(err[bad] / ref["gb"][bad])], np.max(err[bad]), ref["gb"][bad[0]], ref["e"])
    if z is not None:
        err = np.abs((np.asarray(z, dtype=LD) - ref["z"]).astype(np.float64))
        bad = np.nonzero(err > ref["zb"])[0]
        assert len(bad) == 0, "%s: z of %d rows off, worst %.3e" % (what, len(bad), np.max(err))
    if loss is not None:
        err = abs(float(LD(loss) - ref["loss"]))
        assert err <= ref["lb"], "%s: loss off by %.3e > %.3e" % (what, err, ref["lb"])


def csr_case(rng, n, m, lens, kind):
    """rows of the lengths `lens` in turn (at most m), distinct columns (an arithmetic progression mod m with a step
    coprime to m, from a random start), values of the given kind"""
    L = np.minimum(np.asarray(lens, dtype=np.int64)[np.arange(n) % len(lens)], m)
    rowptr = np.concatenate([[0], np.cumsum(L)]).astype(np.int64)
    nnz = int(rowptr[-1])
    rowid = np.repeat(np.arange(n, dtype=np.int64), L)
    k = np.arange(nnz, dtype=np.int64) - rowptr[rowid]
    steps = np.array([s for s in (1, 7, 11, 101, 1009) if math.gcd(s, m) == 1])
    step, start = rng.choice(steps, n), rng.integers(0, max(m, 1), n)
    c = (start[rowid] + k * step[rowid]) % max(m, 1)
    key = np.sort(rowid * m + c)
    col = (key % max(m, 1)).astype(np.int32)
    sign = np.where(rng.random(nnz) < 0.5, -1.0, 1.0)
    if kind == "counts":
        val, vt = rng.integers(1, 6, nnz).astype(np.float64), 3.0
    elif kind == "negreal":
        val, vt = sign * rng.uniform(0.05, 3.0, nnz), 1.5
    elif kind == "tiny":
        val, vt = sign * rng.uniform(1e-9, 1e-6, nnz), 5e-7
    elif kind == "mixed":
        val, vt = rng.integers(1, 6, nnz).astype(np.float64), 3.0
    else:
        raise ValueError(kind)
    theta = rng.normal(scale=1.0 / (vt * math.sqrt(1.0 + float(np.mean(L)) if n else 1.0)), size=m + 1)
    theta[0] = 0.3
    if kind == "mixed" and nnz:
        big = int(np.argmax(np.bincount(col, minlength=m)))
        at = np.nonzero(col == big)[0]
        val[at] = np.where(np.arange(len(at)) % 2 == 0, 1e12, 1e-3)
        theta[big + 1] = 1e-13
    return rowptr, col, val, theta


CYCLE = (0, 1, 31, 32, 33, 1000)
CASES = [  # n, m, row lengths, values, class weights
    (1, 1, (1,), "counts", (1.0, 1.0)),
    (31, 6143, CYCLE, "negreal", (0.7, 1.9)),
    (257, 6144, CYCLE, "tiny", (1e-3, 1e3)),
    (257, 6145, CYCLE, "mixed", (1.0, 1.0)),
    (31, 16385, CYCLE, "counts", (1e-3, 1e3)),
    (257, 70000, CYCLE, "negreal", (1.0, 1.0)),
    (31, 6144, (0,), "counts", (0.7, 1.9)),
    (70001, 70000, CYCLE, "negreal", (0.7, 1.9)),
    (70001, 6145, CYCLE, "tiny", (1e-3, 1e3)),
    (1, 6145, (1000,), "mixed", (0.7, 1.9)),
]


@pytest.mark.parametrize("n,m,lens,kind,cw", CASES, ids=["n%d-m%d-%s-%s" % (c[0], c[1], "x".join(map(str, c[2])), c[3])
                                                          for c in CASES])
def test_imported_gradient_per_column_bound(K, n, m, lens, kind, cw):
    """fused_kernel<double>: hot / cold split, the lo/hi carry of the shared-memory words (negative values), rows
    around a warp, scales far from 1 (tiny values, 1e12 next to 1e-3), empty rows and an empty matrix"""
    rng = np.random.default_rng(n * 7 + m)
    rowptr, col, val, theta = csr_case(rng, n, m, lens, kind)
    y = (rng.random(n) < 0.4).astype(np.uint8)
    if n > 1:
        y[0], y[1] = 1, 0
    d = K.from_csr(n, m, rowptr, col if len(col) else [0], val if len(val) else [0.0])
    try:
        d.SetLabels(y)
        lr = K.logisticRegression(theta, cw)
        ref = reference(n, m, rowptr, col, val, y, theta, cw)
        check_against(ref, g=lr.Gradient(None, d), z=lr.LinearPdf(d), loss=lr.Loss(d), what="imported")
    finally:
        d.free()


# ---------------------------------------------------------------------------------------------------
# tunables that only change the order of the integer additions
# ---------------------------------------------------------------------------------------------------
def _everything(K, d, theta, cw, lam):
    lr = K.logisticRegression(theta, cw)
    g, lo = lr.Gradient(None, d), lr.Loss(d)
    est = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=1e-300, MaxIterations=6)
    est.Theta, est.ClassWeights = theta.copy(), np.array(cw)
    it, delta = est.estimate_proximal(d, lam)
    return g, lo, est.Theta, it, delta, est.hook_state.copy()


def test_order_only_tunables_are_bit_identical(K):
    """hot_cols and fused_ticket move columns between shared memory and L2 and change which warp adds which rows:
    the gradient, the loss and the prox-grad iterates must keep their bits"""
    from kmerlr_b200 import synth
    rng = np.random.default_rng(2)
    n, m = 3000, 20000
    rowptr, col, val, theta_i = csr_case(rng, n, m, CYCLE, "negreal")
    y_i = (rng.random(n) < 0.5).astype(np.uint8)
    di = K.from_csr(n, m, rowptr, col, val)
    di.SetLabels(y_i)
    buf, off, y_c = synth.training_set(400, 400, 150)
    dc = K.compile_test_data(None, K.NewKmerCounter(1, 6, revcomp=True), None, None, True, False, (buf, off))
    dc.SetLabels(y_c)
    assert dc.m > 1023 and di.m > 1023                     # the full-space path of proxgrad
    theta_c = rng.normal(scale=0.01, size=dc.m + 1)
    try:
        K.option("implicit", 0)
        for d, theta, cw, lam in ((di, theta_i, (0.7, 1.9), 1e-3), (dc, theta_c, (0.8, 1.3), 1e-4)):
            first = None
            for hot in (0, 1, 6144, 16384):
                for tk in (0, 1, 8, 4096):
                    K.option("hot_cols", hot)
                    K.option("fused_ticket", tk)
                    r = _everything(K, d, theta, cw, lam)
                    assert r[3] == 6
                    if first is None:
                        first = r
                        continue
                    assert np.array_equal(r[0], first[0]), (hot, tk)
                    assert r[1] == first[1] and np.array_equal(r[2], first[2]) and r[3] == first[3], (hot, tk)
                    assert r[4] == first[4] and np.array_equal(r[5], first[5]), (hot, tk)
    finally:
        restore(K)
        di.free(); dc.free()


# ---------------------------------------------------------------------------------------------------
# power-of-two scale invariance
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [-30, -12, -1, 1, 12, 30])
def test_power_of_two_scale_invariance(K, k):
    """X' = 2^-k X, theta' = (theta_0, 2^k theta_1..): the same z bits, so a scale that tracks max|v| gives
    g'_j = 2^-k g_j exactly; the bias only within its bound (its scale is capped at max|v| = 1)"""
    rng = np.random.default_rng(3)
    n, m = 2000, 7000
    rowptr, col, val, theta = csr_case(rng, n, m, CYCLE, "negreal")
    val = val * (5.0 / 3.0)
    val[len(val) // 2] = 5.0
    assert np.max(np.abs(val)) == 5.0
    y = (rng.random(n) < 0.5).astype(np.uint8)
    cw = (0.7, 1.9)
    vs, ts = np.ldexp(val, -k), theta.copy()
    ts[1:] = np.ldexp(theta[1:], k)
    d, ds = K.from_csr(n, m, rowptr, col, val), K.from_csr(n, m, rowptr, col, vs)
    try:
        d.SetLabels(y); ds.SetLabels(y)
        lr, lrs = K.logisticRegression(theta, cw), K.logisticRegression(ts, cw)
        assert np.array_equal(lr.LinearPdf(d), lrs.LinearPdf(ds))
        assert lr.Loss(d) == lrs.Loss(ds)
        g, gs = lr.Gradient(None, d), lrs.Gradient(None, ds)
        assert np.array_equal(gs[1:], np.ldexp(g[1:], -k)), "columns: %d of %d differ" % (
            int(np.sum(gs[1:] != np.ldexp(g[1:], -k))), m)
        check_against(reference(n, m, rowptr, col, vs, y, ts, cw), g=gs, what="scaled by 2^%d" % -k)
    finally:
        d.free(); ds.free()


# ---------------------------------------------------------------------------------------------------
# above-grid sizes against the oracle (n > 65 536 rows, m > 65 536 columns: every fixed grid strides)
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def big(oracle):
    from kmerlr_b200 import synth
    buf, off, y = synth.training_set(35001, 35000, 120)
    return buf, off, y


def _oracle_close(g, og, lo, olo):
    assert np.max(np.abs(g - og)) <= 1e-10 * np.max(np.abs(og))
    assert abs(lo - olo) <= 1e-12 * abs(olo)


@pytest.mark.parametrize("binarize", [False, True], ids=["counts", "binarized"])
def test_above_grid_sizes_against_oracle(K, oracle, big, binarize):
    buf, off, y = big
    O = oracle
    n = len(off) - 1
    assert n > 65536
    kc, oc = K.NewKmerCounter(1, 9, revcomp=True), O.make_config(1, 9, revcomp=True, binarize=binarize)
    d = K.compile_test_data(None, kc, None, None, True, binarize, (buf, off))
    ref = O.extract(oc, (buf, off), threads=0)
    try:
        assert d.m == ref.m and d.m > 65536 and d.nnz == ref.nnz
        d.SetLabels(y)
        cw = K.compute_class_weights(y)
        assert np.array_equal(d.class_weights(), cw)
        rowptr, col, val = ref.rows()
        theta = np.random.default_rng(4).normal(scale=0.003, size=d.m + 1)
        lr = K.logisticRegression(theta, cw)
        R = reference(n, d.m, rowptr, col, val, y, theta, cw)
        del rowptr, col, val
        og, olo = O.gradient(ref, y, theta, cw), O.loss(ref, y, theta, cw)
        lo = lr.Loss(d)
        check_against(R, z=lr.LinearPdf(d), loss=lo, what="extraction")
        paths = (1, 0) if not binarize else (1,)
        for implicit in paths:                             # matrix-free pass, then the pass over the stored rows
            K.option("implicit", implicit)
            g = lr.Gradient(None, d)
            check_against(R, g=g, what="implicit=%d" % implicit)
            _oracle_close(g, og, lo, olo)
        if binarize:
            return
        # from theta = 0 the loss falls by 8.30e-6, 8.26e-6 (8th), 8.24e-6 (12th), ... per iteration: 8.25e-6 stops
        # the run near the 10th, with 5e-9 between neighbouring decrements (an oracle iteration costs 0.4 s here)
        lam = 2e-4
        for eps_loss, cap in ((0.0, 8), (8.25e-6, 100000)):
            oth, oit, _ = O.proxgrad(ref, y, np.zeros(d.m + 1), cw, lam=lam, epsilon=0.0, epsilon_loss=eps_loss,
                                     max_iter=cap)
            if cap == 8:
                assert oit == 8
            else:
                assert 1 < oit < cap
            for implicit in paths:
                K.option("implicit", implicit)
                est = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=eps_loss, MaxIterations=cap)
                est.Theta, est.ClassWeights = np.zeros(d.m + 1), cw
                it, _ = est.estimate_proximal(d, lam)
                assert it == oit, (implicit, eps_loss, it, oit)
                assert np.max(np.abs(est.Theta - oth)) <= 1e-9, (implicit, eps_loss)
                assert np.array_equal(est.Theta == 0.0, oth == 0.0)
    finally:
        restore(K)
        d.free()


# ---------------------------------------------------------------------------------------------------
# labels normalised on the device
# ---------------------------------------------------------------------------------------------------
def test_labels_normalised_on_the_device(K):
    """n = 200 001 rows: more than one grid stride of normalize_labels.  Any non-zero byte is a positive label"""
    rng = np.random.default_rng(5)
    n, m = 200001, 2000
    rowptr, col, val, theta = csr_case(rng, n, m, (0, 1, 3, 7), "counts")
    y = (rng.random(n) < 0.3).astype(np.uint8)
    raw = np.where(y == 1, rng.choice(np.array([1, 2, 128, 255], dtype=np.uint8), n), 0).astype(np.uint8)
    assert set(np.unique(raw).tolist()) == {0, 1, 2, 128, 255}
    cw_ref = K.compute_class_weights(y)
    d = K.from_csr(n, m, rowptr, col, val)
    try:
        out = {}
        for name, lab in (("raw", raw), ("01", y), ("raw again", raw)):
            d.SetLabels(lab)
            cw = d.class_weights()
            assert np.array_equal(cw, cw_ref), name
            lr = K.logisticRegression(theta, cw)
            out[name] = (lr.Gradient(None, d), lr.Loss(d))
        for name in ("raw", "raw again"):
            assert np.array_equal(out[name][0], out["01"][0]) and out[name][1] == out["01"][1], name
    finally:
        d.free()


# ---------------------------------------------------------------------------------------------------
# device top-2N select (KMERLR_TIE_INDEX) against the host path
# ---------------------------------------------------------------------------------------------------
def select_restated(g, N):
    """select_core (select.cu) for an empty active set, in numpy: |g| descending, index ascending"""
    a = np.abs(g[1:])
    order = np.lexsort((np.arange(len(a)), -a))
    top = min(len(a), 2 * N)
    cand = order[:top]
    new = cand[g[1:][cand] != 0.0][:N]
    old = cand[g[1:][cand] == 0.0][:N - len(new)]
    b = np.zeros(len(g), dtype=bool)
    b[0] = True
    b[new + 1] = True
    b[old + 1] = True
    lam = 0.0
    if N <= top:
        v = a[order[N - 1]]
        below = a[a < v]
        lam = (v + (below.max() if len(below) else 0.0)) / 2.0
    return b, lam, len(new) > 0


def test_device_select_ties_across_blocks(K):
    """m = 300 000 columns, each a copy of one of four base columns or empty: integer sums give copies the same bits,
    so every copy group is an exact tie group spread over all blocks of the radix select.  The cut inside a tie group,
    a tie group filling every top place (lambda from device_max_below), 2N >= m, lambda = 0"""
    rng = np.random.default_rng(6)
    n, m = 64, 300000
    y = np.zeros(n, dtype=np.uint8)
    y[rng.permutation(n)[:32]] = 1
    pos, neg = np.nonzero(y == 1)[0], np.nonzero(y == 0)[0]
    bases = [  # (rows, values): |g| = 8, 4 (plus and minus: one tie group), 2 units of 0.5 / n; the rest empty
        (pos[4:8], 2.0), (pos[0:4], 1.0), (neg[0:4], 1.0), (np.concatenate([pos[8:11], neg[4:5]]), 1.0)]
    sizes = [40000, 50000, 50000, 100000]
    group = np.full(m, -1)
    perm = rng.permutation(m)
    at = 0
    for b, s in enumerate(sizes):
        group[perm[at:at + s]] = b
        at += s
    cols_of = [np.nonzero(group == b)[0] for b in range(len(bases))]
    rows, cols = [], []
    for (r, _), cs in zip(bases, cols_of):
        rr, cc = np.meshgrid(r, cs, indexing="ij")
        rows.append(rr.ravel()); cols.append(cc.ravel())
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    vals = np.concatenate([np.full(len(r) * len(cs), v) for (r, v), cs in zip(bases, cols_of)])
    o = np.lexsort((cols, rows))
    rows, cols, vals = rows[o], cols[o], vals[o]
    rowptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=n))])
    d = K.from_csr(n, m, rowptr, cols.astype(np.int32), vals)
    try:
        d.SetLabels(y)
        cw = (1.0, 1.0)
        for N in (2, 5000, 30000, 45000, 150000, 200000, 270000):
            fs = K.featureSelector(cw, False, N, m, tie=K.TIE_INDEX)
            dev, lam_d, ok_d = fs.Select(d, 0.0, [], [], 0.0)
            host, lam_h, ok_h = fs.Select(d, 0.0, [], [], 0.0, want_gradient=True)
            g = host.g
            if N == 2:                                     # the tie groups are what the test is about
                for b, cs in enumerate(cols_of):
                    assert len(set(g[cs + 1].tolist())) == 1, b
                assert g[cols_of[1][0] + 1] == -g[cols_of[2][0] + 1] != 0.0
                assert np.all(g[1:][group == -1] == 0.0)
            assert np.array_equal(dev.b, host.b) and lam_d == lam_h and ok_d == ok_h and dev.c == host.c, N
            b, lam, ok = select_restated(g, N)
            assert np.array_equal(host.b, b) and lam_h == lam and ok_h == ok, N
    finally:
        d.free()
