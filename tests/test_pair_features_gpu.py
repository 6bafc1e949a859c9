"""Pair features (Cooccurrence) at the C4 scale of BASELINE: k = 1..6 revcomp, m = 2 772 columns, 3 843 379
coefficients, the 16 000 training rows of fold 0 (fold = i mod 5 over fg || bg, as bench.py's leg_c4 takes them).

- the blocked pair gradient (pairs_gradient) adds (w v_a) v_b in sample order: the bits of the serial loop, over all
  63 chunks of 256 rows and all 3 828 tile pairs, for u32 counts, binarized rows and f64 rows; at a general theta it
  stays within a computed error bound that dropping one row or the last partial chunk breaks
- a shape sweep of pairs_gradient around its chunk (256 rows) and tile (32 columns) edges
- the single-feature block of pair mode against the plain gradient
- the row pass on both sides of PAIR_TERMS_MAX (sparse pair terms / the O(q^2) pass) and the zero scan's edges
- pair moments (exact integer sums), pair columns of reduce, Select over the pair space with its tie groups, and
  fold subsets

References are fp64 on the device (torch): one row per step in the serial order where bits are compared, dense
float64 products with an error bound elsewhere."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -53
DEV = "cuda"
N_SEQ, LEN = 10000, 500
CW = (0.8, 1.3)
THETA0 = -0.4


def ind2sub(m, a, b):
    """CoeffIndex(m).Ind2Sub(a, b) for a < b (numpy or torch int64)"""
    return m + m * (m - 1) // 2 - (m - a) * (m - a - 1) // 2 + b - a


def coeff_dim(m):
    return (m + 1) * m // 2 + 1


def dense(rows, n, m):
    rp, col, val = rows
    X = torch.zeros((n, m), dtype=torch.float64, device=DEV)
    r = torch.repeat_interleave(torch.arange(n, device=DEV), torch.as_tensor(np.diff(rp), device=DEV))
    X[r, torch.as_tensor(col.astype(np.int64), device=DEV)] = torch.as_tensor(val, device=DEV)
    return X


def take_rows(rows, idx):
    rp, col, val = rows
    parts = [np.arange(rp[i], rp[i + 1]) for i in idx]
    p = np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)
    return np.concatenate([[0], np.cumsum(np.diff(rp)[idx])]).astype(np.int64), col[p], val[p]


def log_add0(x):
    return np.where(x > 0.0, x + np.log1p(np.exp(-np.abs(x))), np.log1p(np.exp(np.minimum(x, 0.0))))


def host_w(z, y, cw, n):
    """the row weight of kmerLr_logistic_regression.go:166-178 from z, in fp64 on the host"""
    r = -log_add0(-z)
    inv_n = 1.0 / n
    return np.where(y == 1, inv_n * cw[1] * (np.exp(r) - 1.0), inv_n * cw[0] * np.exp(r))


def serial_pair_gradient(rows, m, w):
    """g[Ind2Sub(a, b)] += (w_i v_ia) v_ib for a < b, row after row (the reference's serial loop): every product and
    every addition a separate fp64 rounding.  Pairs of one row have distinct indices, so index_add_ adds each once."""
    rp, col, val = rows
    n = len(rp) - 1
    c = torch.as_tensor(col.astype(np.int64), device=DEV)
    v = torch.as_tensor(val, dtype=torch.float64, device=DEV)
    wt = torch.as_tensor(np.asarray(w, dtype=np.float64), device=DEV)
    G = torch.zeros(coeff_dim(m), dtype=torch.float64, device=DEV)
    for i in range(n):
        a, b = int(rp[i]), int(rp[i + 1])
        if b - a < 2:
            continue
        ia, ib = torch.triu_indices(b - a, b - a, 1, device=DEV)
        ci, vi = c[a:b], v[a:b]
        G.index_add_(0, ind2sub(m, ci[ia], ci[ib]), (wt[i] * vi[ia]) * vi[ib])
    return G.cpu().numpy()


def bias_weights(K, y, theta0, cw):
    """(w_+, w_-) as the device computes them at theta = bias only (z = theta_0 on every row): a probe matrix with the
    same n and labels whose pair (0, 1) lives in one positive row and pair (2, 3) in one negative row only"""
    n = len(y)
    pos, neg = np.nonzero(y == 1)[0], np.nonzero(y == 0)[0]
    per = np.zeros(n, dtype=np.int64)
    cols = {}
    if len(pos):
        per[pos[0]] = 2; cols[pos[0]] = [0, 1]
    if len(neg):
        per[neg[0]] = 2; cols[neg[0]] = [2, 3]
    col = np.array([c for i in sorted(cols) for c in cols[i]] or [0], dtype=np.int32)
    p = K.from_csr(n, 4, np.concatenate([[0], np.cumsum(per)]), col, np.ones(len(col)))
    try:
        p.SetLabels(y)
        t = np.zeros(coeff_dim(4))
        t[0] = theta0
        g = K.logisticRegression(t, cw, 0.0, Cooccurrence=True).Gradient(None, p)
    finally:
        p.free()
    return g[ind2sub(4, 0, 1)], g[ind2sub(4, 2, 3)]


def pair_theta(m, singles, pairs, rng, theta0=THETA0, s_scale=2e-3, p_scale=2e-4):
    t = np.zeros(coeff_dim(m))
    t[0] = theta0
    if singles:
        t[1:m + 1] = rng.normal(scale=s_scale, size=m)
    if pairs:
        idx = rng.choice(coeff_dim(m) - (m + 1), size=pairs, replace=False) + m + 1
        t[idx] = rng.normal(scale=p_scale, size=pairs)
    return t


def upper(theta, m):
    """the pair coefficients as a strictly upper triangular m x m matrix U (U[a, b] = theta[Ind2Sub(a, b)])"""
    U = torch.zeros((m, m), dtype=torch.float64, device=DEV)
    iu = torch.triu_indices(m, m, 1, device=DEV)
    U[iu[0], iu[1]] = torch.as_tensor(theta[m + 1:], device=DEV)
    return U


def model_reference(X, theta, q_max, nterms):
    """z = theta_0 + X theta_s + sum_{a<b} v_a v_b theta_ab (rowwise sum of (X U) o X) with the allowed error of every
    z_i: 4 (K + 2) u times the sum of the absolute terms, K = the terms either side sums (the reference's products over
    m, the device's q singles and its pair terms)"""
    n, m = X.shape
    th = torch.as_tensor(theta, device=DEV)
    U, A = upper(theta, m), X.abs()
    z = th[0] + X @ th[1:m + 1] + ((X @ U) * X).sum(1)
    Z = th[0].abs() + A @ th[1:m + 1].abs() + ((A @ U.abs()) * A).sum(1)
    k = 2 * m + max(q_max * (q_max - 1) // 2, nterms) + 2
    return z.cpu().numpy(), 4.0 * (k + 2) * EPS * Z.cpu().numpy()


def gradient_bound(X, w, dw):
    """per-entry bound of |g_device - g_reference| for g = X^T w (singles) and X^T diag(w) X (pairs): 4 (n + 2) u times
    the sum of |terms| for the two summation orders, plus sum_i dw_i |x_ia x_ib| for the error of w"""
    n = X.shape[0]
    A = X.abs()
    aw, dw = torch.as_tensor(np.abs(w), device=DEV), torch.as_tensor(dw, device=DEV)
    c = 4.0 * (n + 2) * EPS
    return c * (A.T @ aw) + A.T @ dw, c * (A.T @ (A * aw[:, None])) + A.T @ (A * dw[:, None])


def pairs_of(Mx):
    """the entries a < b of an m x m matrix in CoeffIndex order"""
    m = Mx.shape[0]
    iu = torch.triu_indices(m, m, 1, device=Mx.device)
    return Mx[iu[0], iu[1]].cpu().numpy()


def fixed_point_bound(vmax, cw, n):
    """what the fixed-point single-feature gradient may lose: half a unit of 2^-e per term (logistic.cu set_scale)"""
    e = 60 - int(np.ceil(np.log2(max(abs(cw[0]), abs(cw[1])) * max(vmax, 1.0))))
    return (0.5 * n + 1.0) * 2.0 ** -e


def check_model(K, d, X, y, theta, cw, nterms, what):
    """LinearPdf, LogPdf, Loss and Gradient of pair mode against the dense reference within their bounds.  The reference
    gradient takes w from the reference z on the host; its allowed error per row is the z bound through
    dw/dz <= cw / (4 n) plus 8 u cw / n for the last bits of exp and log.  Returns (device gradient, bound of every
    entry, reference w, dw)."""
    n, m = X.shape
    q_max = int((X != 0).sum(1).max().item())
    lr = K.logisticRegression(theta, cw, 0.0, Cooccurrence=True)
    z = lr.LinearPdf(d)
    zr, zb = model_reference(X, theta, q_max, nterms)
    bad = np.abs(z - zr) > zb
    assert not bad.any(), "%s: z of %d rows off, worst %.3e" % (what, bad.sum(), np.max(np.abs(z - zr)))
    lp = lr.LogPdf(d)
    lpr = -log_add0(-zr)
    assert np.all(np.abs(lp - lpr) <= zb + 8 * EPS * (np.abs(lpr) + 1.0)), what
    cwy = np.where(y == 1, cw[1], cw[0])
    lo = lr.Loss(d)
    lref = np.where(y == 1, cw[1] * log_add0(-zr), cw[0] * log_add0(zr)).sum() / n
    lb = np.sum(cwy * zb) / n + 1e-13 * abs(lref)
    assert abs(lo - lref) <= lb, "%s: loss %.17g vs %.17g" % (what, lo, lref)
    g = lr.Gradient(None, d)
    w = host_w(zr, y, cw, n)
    dw = cwy / n * (zb / 4.0 + 8.0 * EPS)
    wt = torch.as_tensor(w, device=DEV)
    sb, pb = gradient_bound(X, w, dw)
    ref = np.concatenate([[wt.sum().item()], (X.T @ wt).cpu().numpy(), pairs_of(X.T @ (X * wt[:, None]))])
    bound = np.concatenate([[4.0 * (n + 2) * EPS * np.abs(w).sum() + dw.sum()], sb.cpu().numpy(), pairs_of(pb)])
    bound[:m + 1] += fixed_point_bound(float(X.abs().max()), cw, n)
    err = np.abs(g - ref)
    bad = np.nonzero(err > bound)[0]
    assert len(bad) == 0, "%s: %d gradient entries off (%d singles), worst %.3e at %d (bound %.3e)" % (
        what, len(bad), np.sum(bad <= m), err[bad].max(), bad[np.argmax(err[bad])], bound[bad[np.argmax(err[bad])]])
    return g, bound, w, dw


# ---------------------------------------------------------------------------------------------------
# the C4 data: training rows of fold 0, counts and binarized, and the f64 copy of the counts rows
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def c4(K):
    from kmerlr_b200 import synth
    buf, off, y = synth.training_set(N_SEQ, N_SEQ, LEN)
    n = len(off) - 1
    tr = np.nonzero(np.arange(n) % 5 != 0)[0]
    lens = np.diff(off)
    o = np.concatenate([[0], np.cumsum(lens[tr])]).astype(np.int64)
    b = np.concatenate([buf[off[i]:off[i + 1]] for i in tr])
    kc = K.NewKmerCounter(1, 6, revcomp=True)
    dc = K.compile_test_data(None, kc, None, None, True, False, (b, o))
    db = K.compile_test_data(None, kc, None, None, True, True, (b, o))
    yt = y[tr].astype(np.uint8)
    dc.SetLabels(yt); db.SetLabels(yt)
    assert dc.n == db.n == 16000 and dc.m == db.m == 2772 and coeff_dim(dc.m) == 3843379
    rc, rb = dc.rows(), db.rows()
    df = K.from_csr(dc.n, dc.m, *rc)
    df.SetLabels(yt)
    data = dict(counts=dc, binarized=db, f64=df, rows=dict(counts=rc, binarized=rb, f64=rc), y=yt, tr=tr,
                seqs=(buf, off, y), X={})
    yield data
    for h in (dc, db, df):
        h.free()
    data["X"].clear()
    torch.cuda.empty_cache()


def X_of(c4, kind):
    if kind not in c4["X"]:
        c4["X"][kind] = dense(c4["rows"][kind], 16000, 2772)
    return c4["X"][kind]


# ---------------------------------------------------------------------------------------------------
# 1. the pair gradient is the serial loop's bits
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["counts", "binarized", "f64"])
def test_pair_gradient_is_the_serial_loop_at_c4(K, c4, kind):
    d, y, m = c4[kind], c4["y"], 2772
    wp, wm = bias_weights(K, y, THETA0, CW)
    assert wp < 0.0 < wm
    t = np.zeros(coeff_dim(m))
    t[0] = THETA0
    g = K.logisticRegression(t, CW, 0.0, Cooccurrence=True).Gradient(None, d)
    ref = serial_pair_gradient(c4["rows"][kind], m, np.where(y == 1, wp, wm))
    bad = np.nonzero(g[m + 1:] != ref[m + 1:])[0]
    assert len(bad) == 0, "%s: %d of %d pair entries differ, first at %d" % (kind, len(bad), len(ref) - m - 1, bad[0])
    assert np.count_nonzero(ref[m + 1:]) > 10 ** 6


# ---------------------------------------------------------------------------------------------------
# 2. a general theta: within the error bound, which one dropped row or the dropped last chunk breaks
# ---------------------------------------------------------------------------------------------------
def test_pair_gradient_general_theta_within_bound(K, c4):
    """non-zero singles and 300 pairs (the shape of theta after a first leapfrog epoch): the sparse-term row pass, then
    the blocked gradient against X^T diag(w) X.  The same bound must notice a reference without the last partial
    chunk (rows 15 872..15 999) or without one row."""
    d, y, m = c4["counts"], c4["y"], 2772
    X = X_of(c4, "counts")
    theta = pair_theta(m, True, 300, np.random.default_rng(11))
    g, bound, w, _ = check_model(K, d, X, y, theta, CW, 300, "general theta")
    wt = torch.as_tensor(w, device=DEV)
    assert 15872 == 62 * 256 and d.n - 15872 == 128
    for what, keep in (("last partial chunk", np.arange(15872)), ("one row", np.r_[0:7000, 7001:d.n])):
        keep = torch.as_tensor(keep, device=DEV)
        Xk, wk = X[keep], wt[keep]
        gp = pairs_of(Xk.T @ (Xk * wk[:, None]))
        assert np.any(np.abs(g[m + 1:] - gp) > bound[m + 1:]), "the bound does not notice a dropped %s" % what


# ---------------------------------------------------------------------------------------------------
# 3. shape sweep of pairs_gradient (chunk edges at 256 rows, tile edges at 32 columns)
# ---------------------------------------------------------------------------------------------------
def sweep_case(rng, n, m, kind):
    """random rows of about 10 % density plus: one dense row (all columns but the empty one), an empty column, a column
    whose entries lie only in the last partial chunk, a column with an entry in every chunk"""
    P = rng.random((n, m)) < 0.1
    P[n - 1, :] = True                                          # one dense row (in the last chunk)
    if m > 4:
        P[:, 2] = False                                        # empty
        P[:, m - 1] = False
        P[(n - 1) // 256 * 256:, m - 1] = True                  # last (partial) chunk only
        P[::256, 1] = True                                      # every chunk
    if kind == "counts":
        V = rng.integers(1, 40, (n, m)).astype(np.float64)
    elif kind == "large":
        V = rng.integers(1, 10 ** 6 + 1, (n, m)).astype(np.float64)
    else:
        V = rng.normal(scale=3.0, size=(n, m)) * 10.0 ** rng.integers(-3, 3, (n, m))
    V = np.where(P, V, 0.0)
    rp = np.concatenate([[0], np.cumsum(P.sum(1))]).astype(np.int64)
    r, c = np.nonzero(P)
    return (rp, c.astype(np.int32), V[r, c]), P


@pytest.mark.parametrize("kind", ["counts", "large", "real"])
@pytest.mark.parametrize("n,m", [(1, 2), (20, 70), (255, 32), (256, 33), (257, 64), (513, 65), (1100, 690)])
def test_pair_gradient_shape_sweep(K, n, m, kind):
    rng = np.random.default_rng(1000 * n + m)
    rows, _ = sweep_case(rng, n, m, kind)
    y = (rng.random(n) < 0.5).astype(np.uint8)
    y[0] = 1
    if n > 1:
        y[1] = 0
    d = K.from_csr(n, m, *rows)
    try:
        d.SetLabels(y)
        wp, wm = bias_weights(K, y, 0.3, (0.7, 1.9))
        t = np.zeros(coeff_dim(m))
        t[0] = 0.3
        g = K.logisticRegression(t, (0.7, 1.9), 0.0, Cooccurrence=True).Gradient(None, d)
        ref = serial_pair_gradient(rows, m, np.where(y == 1, wp, wm))
        bad = np.nonzero(g[m + 1:] != ref[m + 1:])[0]
        assert len(bad) == 0, "%d pair entries differ, first %s" % (len(bad), bad[:4])
        if m > 4:
            a = np.arange(m)
            assert np.all(g[ind2sub(m, np.minimum(a[a != 2], 2), np.maximum(a[a != 2], 2))] == 0.0)
    finally:
        d.free()


# ---------------------------------------------------------------------------------------------------
# 4. the single-feature block of pair mode
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["counts", "binarized"])
def test_single_block_of_pair_mode(K, c4, kind):
    d, m = c4[kind], 2772
    t = np.zeros(coeff_dim(m))
    t[0] = THETA0
    g = K.logisticRegression(t, CW, 0.0, Cooccurrence=True).Gradient(None, d)
    try:
        K.option("implicit", 0)
        g0 = K.logisticRegression(t[:m + 1], CW, 0.0).Gradient(None, d)
        K.option("implicit", 1)
        g1 = K.logisticRegression(t[:m + 1], CW, 0.0).Gradient(None, d)
    finally:
        K.option("implicit", 1)
    assert np.array_equal(g[:m + 1], g0)
    # the matrix-free pass adds count x round(w S) where the row pass adds round(w S v): each may lose half a unit of
    # 2^-e per entry and per unit of the count (the bound of the matrix-free tests in test_gradient_edges_gpu.py)
    _, col, val = c4["rows"][kind]
    per = np.bincount(col, weights=np.maximum(1.0, val), minlength=m)
    e = 60 - int(np.ceil(np.log2(max(CW) * max(float(val.max()), 1.0))))
    bound = 2.0 ** -e * (np.concatenate([[0.5 * d.n], per]) + 2.0)
    assert np.all(np.abs(g1 - g0) <= bound)


# ---------------------------------------------------------------------------------------------------
# 5. the row pass on both sides of PAIR_TERMS_MAX = 8 192 and the edges of the zero scan
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def small(K, c4):
    """the first 2 000 training rows as an f64 matrix (the dense-theta pass is O(q^2) per row)"""
    rows = take_rows(c4["rows"]["counts"], np.arange(2000))
    d = K.from_csr(2000, 2772, *rows)
    y = c4["y"][:2000]
    d.SetLabels(y)
    yield d, dense(rows, 2000, 2772), y
    d.free()


@pytest.mark.parametrize("pairs", [0, 1, 8192, 8193, 50000, "all"])
def test_row_pass_both_sides_of_pair_terms_max(K, small, pairs):
    d, X, y = small
    m = 2772
    rng = np.random.default_rng(7)
    if pairs == "all":
        theta = pair_theta(m, True, 0, rng, p_scale=1e-6)
        theta[m + 1:] = rng.normal(scale=1e-6, size=coeff_dim(m) - m - 1)
        theta[m + 1:][theta[m + 1:] == 0.0] = 1e-7
        nterms = coeff_dim(m) - m - 1
    else:
        theta = pair_theta(m, True, pairs, rng, p_scale=2e-5)
        nterms = pairs
    assert np.count_nonzero(theta[m + 1:]) == nterms
    check_model(K, d, X, y, theta, CW, nterms, "%s pair terms" % pairs)


@pytest.mark.parametrize("where", ["first", "last"] + ["offset%d" % o for o in range(8)])
def test_zero_scan_single_nonzero(K, small, where):
    d, X, y = small
    m = 2772
    nt = coeff_dim(m)
    if where == "first":
        j = m + 1
    elif where == "last":
        j = nt - 1
    else:                                                      # offset o of the fourth eight-block of the scan
        j = m + 1 + 8 * 3 + int(where[len("offset"):])
    theta = np.zeros(nt)
    theta[0] = THETA0
    theta[j] = 1e-3
    a, b = K.CoeffIndex(m).Sub2Ind(j - 1)
    assert (X[:, a] * X[:, b] != 0).any(), "pair (%d, %d) in no row" % (a, b)
    check_model(K, d, X, y, theta, CW, 1, where)


def test_zero_scan_negative_zeros(K, small):
    """-0.0 is a zero of theta: 8 192 non-zeros plus thousands of -0.0 stay on the sparse-term path with the same bits"""
    d, X, y = small
    m = 2772
    rng = np.random.default_rng(8)
    theta = pair_theta(m, True, 8192, rng, p_scale=2e-5)
    tz = theta.copy()
    zeros = np.nonzero(tz[m + 1:] == 0.0)[0] + m + 1
    tz[rng.choice(zeros, 5000, replace=False)] = -0.0
    tz[zeros[:8]] = -0.0                                       # one whole eight-block of -0.0 at the scan's start
    tz[coeff_dim(m) - 3:] = np.where(tz[coeff_dim(m) - 3:] == 0.0, -0.0, tz[coeff_dim(m) - 3:])
    assert np.sum(np.signbit(tz) & (tz == 0.0)) >= 5000
    a = K.logisticRegression(theta, CW, 0.0, Cooccurrence=True)
    b = K.logisticRegression(tz, CW, 0.0, Cooccurrence=True)
    assert np.array_equal(a.LinearPdf(d), b.LinearPdf(d))
    assert np.array_equal(a.LogPdf(d), b.LogPdf(d))
    assert a.Loss(d) == b.Loss(d)
    assert np.array_equal(a.Gradient(None, d), b.Gradient(None, d))


# ---------------------------------------------------------------------------------------------------
# 6. pair moments: exact integer sums
# ---------------------------------------------------------------------------------------------------
def pair_moments(K, d):
    from kmerlr_b200 import _lib
    npairs = d.m * (d.m - 1) // 2
    s1, s2, mx = np.zeros(npairs), np.zeros(npairs), np.zeros(npairs)
    cnt = np.zeros(npairs, dtype=np.int64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    _lib.check(_lib.lib().kmerlr_pair_moments(d.h, p(s1), p(s2), p(mx), p(cnt)))
    return s1, s2, mx, cnt


def exact_moments(X):
    """X^T X, (X o X)^T (X o X) and B^T B (B = [X != 0]) in fp64: integer partial sums below 2^53 are exact in any order"""
    B = (X != 0).to(torch.float64)
    X2 = X * X
    assert float(X2.max()) * float(X2.max()) * X.shape[0] < 2.0 ** 53
    return pairs_of(X.T @ X), pairs_of(X2.T @ X2), pairs_of(B.T @ B)


@pytest.mark.parametrize("kind", ["counts", "binarized"])
def test_pair_moments_exact(K, c4, kind):
    d = c4[kind]
    X = X_of(c4, kind)
    s1, s2, mx, cnt = pair_moments(K, d)
    r1, r2, rc = exact_moments(X)
    assert np.array_equal(s1, r1) and np.array_equal(s2, r2) and np.array_equal(cnt, rc.astype(np.int64))
    # the max over a subset of 2 000 rows: the running maximum of the outer products v v^T
    sub = d.subset(np.arange(2000))
    try:
        t1, t2, tm, tc = pair_moments(K, sub)
        Xs = X[:2000]
        q1, q2, qc = exact_moments(Xs)
        assert np.array_equal(t1, q1) and np.array_equal(t2, q2) and np.array_equal(tc, qc.astype(np.int64))
        M = torch.zeros((2772, 2772), dtype=torch.float64, device=DEV)
        for i in range(0, 2000, 16):
            M = torch.maximum(M, (Xs[i:i + 16, :, None] * Xs[i:i + 16, None, :]).amax(0))
        assert np.array_equal(tm, pairs_of(M))
    finally:
        sub.free()
    if kind == "binarized":
        assert np.array_equal(mx, (cnt > 0).astype(np.float64))


def test_pair_moments_far_down_the_triangle(K):
    """m > 6 000 columns (k = 1..7): the decoding of the pair index by sqrt and its two correction loops, pair indices
    up to 3.3e7"""
    from kmerlr_b200 import synth
    buf, off, _ = synth.training_set(15, 15, 300)
    d = K.compile_test_data(None, K.NewKmerCounter(1, 7, revcomp=True), None, None, True, False, (buf, off))
    try:
        assert d.m > 6000
        s1, _, _, cnt = pair_moments(K, d)
        X = dense(d.rows(), d.n, d.m)
        r1, _, rc = exact_moments(X)
        assert np.array_equal(s1, r1) and np.array_equal(cnt, rc.astype(np.int64))
        del X, r1, rc, s1, cnt
    finally:
        d.free()
        torch.cuda.empty_cache()


def test_pair_moments_refuse_f64(K, c4):
    from kmerlr_b200 import _lib
    with pytest.raises(K.KmerLrError) as e:
        pair_moments(K, c4["f64"])
    assert e.value.code == _lib.ERR_ARG


def test_transform_fit_with_pairs_at_c4(K, c4):
    """TransformFull.Fit(cooccurrence=True) = the numpy formulas on the exact moments"""
    d, X = c4["counts"], X_of(c4, "counts")
    r1, r2, _ = exact_moments(X)
    s1 = np.concatenate([X.sum(0).cpu().numpy(), r1])
    s2 = np.concatenate([(X * X).sum(0).cpu().numpy(), r2])
    n = float(d.n)
    t = K.TransformFull().Fit(d, "standardizer", cooccurrence=True)
    mean = s1 / n
    sj = np.maximum(s2 - n * mean * mean, 0.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        sc = np.where(sj == 0.0, 1.0, 1.0 / np.sqrt(sj / (n - 1.0)))
    assert len(t.Offset) == coeff_dim(d.m)
    assert np.array_equal(t.Offset[1:], mean) and np.array_equal(t.Scale[1:], sc)
    t = K.TransformFull().Fit(d, "mean-scaler", cooccurrence=True)
    with np.errstate(divide="ignore"):
        assert np.array_equal(t.Scale[1:], n / s1)


# ---------------------------------------------------------------------------------------------------
# 7. pair columns of kmerlr_reduce
# ---------------------------------------------------------------------------------------------------
def test_reduce_pair_columns(K, c4):
    d, y, m = c4["counts"], c4["y"], 2772
    X = X_of(c4, "counts")
    pairs = [(0, 1), (5, 30), (31, 32), (3, 40), (100, 2000), (2700, 2771), (m - 2, m - 1)]
    singles = [0, 7, 1500, m - 1]
    sel = np.array(sorted([0] + [s + 1 for s in singles] + [ind2sub(m, a, b) for a, b in pairs]), dtype=np.int64)
    r = K.select_data(d, sel)
    try:
        cols = []
        for j in sel[1:]:
            a, b = K.CoeffIndex(m).Sub2Ind(int(j) - 1)
            cols.append(X[:, a] if a == b else X[:, a] * X[:, b])
        R = torch.stack(cols, 1)
        got = dense(r.rows(), d.n, len(sel) - 1)
        assert torch.equal(got, R)
        rng = np.random.default_rng(12)
        tr = np.concatenate([[THETA0], rng.normal(scale=1e-4, size=len(sel) - 1)])
        tf = np.zeros(coeff_dim(m))
        tf[sel] = tr
        gp, bound, w, dw = check_model(K, d, X, y, tf, CW, len(pairs), "embedded theta")
        # the reduced model against the same reference (w of the reference z), with the bound of its fixed-point pass
        lr = K.logisticRegression(tr, CW, 0.0)
        g = lr.Gradient(None, r)
        wt = torch.as_tensor(w, device=DEV)
        ref = np.concatenate([[wt.sum().item()], (R.T @ wt).cpu().numpy()])
        sb, _ = gradient_bound(R, w, dw)
        tol = np.concatenate([[4.0 * (d.n + 2) * EPS * np.abs(w).sum() + dw.sum()], sb.cpu().numpy()])
        tol += fixed_point_bound(float(R.abs().max()), CW, d.n)
        assert np.all(np.abs(g - ref) <= tol)
        assert np.all(np.abs(g - gp[sel]) <= tol + bound[sel])
        lo = K.logisticRegression(tf, CW, 0.0, Cooccurrence=True).Loss(d)
        assert abs(lr.Loss(r) - lo) <= 1e-12 * abs(lo)
    finally:
        r.free()


# ---------------------------------------------------------------------------------------------------
# 8. Select over the pair space (binarized C4: the pairs of the k = 1..3 classes tie exactly at the top)
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


def test_select_over_pairs_at_c4(K, c4, oracle):
    d, m, N = c4["binarized"], 2772, 20
    theta0 = 1.5
    fs = K.featureSelector(CW, True, N, m, tie=K.TIE_INDEX)
    dev, lam_d, ok_d = fs.Select(d, theta0, [], [], 0.0)
    host, lam_h, ok_h = fs.Select(d, theta0, [], [], 0.0, want_gradient=True)
    g = host.g
    assert np.array_equal(dev.b, host.b) and lam_d == lam_h and ok_d == ok_h and dev.c == host.c
    b, lam, ok = select_restated(g, N)
    assert np.array_equal(host.b, b) and lam_h == lam and ok_h == ok
    # the tie group at the cut: every single and pair of the k = 1..3 classes (present in every row)
    v = np.sort(np.abs(g[1:]))[::-1][N - 1]
    assert np.sum(np.abs(g[1:]) == v) > 2 * N
    # warm start with pair coefficients in the active set (the sparse-term row pass)
    ci = K.CoeffIndex(m)
    ai = np.array([6, ci.Ind2Sub(0, 1), ci.Ind2Sub(10, 300), ci.Ind2Sub(40, 2500), ci.Ind2Sub(m - 2, m - 1)], dtype=np.int64)
    at = np.array([0.01, -0.002, 0.003, 0.0, 0.004])
    dev, lam_d, ok_d = fs.Select(d, theta0, ai, at, lam_h)
    host, lam_h2, ok_h = fs.Select(d, theta0, ai, at, lam_h, want_gradient=True)
    assert np.array_equal(dev.b, host.b) and lam_d == lam_h2 and ok_d == ok_h and dev.c == host.c
    o = oracle.select_from_gradient(host.g, N, ai, at, tie=oracle.TIE_INDEX)
    assert np.array_equal(host.b, o["mask"]) and lam_h2 == o["lam"] and ok_h == o["ok"] and host.c == o["c"]
    # TIE_GO118 on the device gradient: the order of Go's sort.Sort
    from kmerlr_b200 import _lib
    nt = len(g)
    mask = np.zeros(nt, dtype=np.uint8)
    lam, c, okc = C.c_double(), C.c_int64(), C.c_int()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    e = np.zeros(1, dtype=np.int64)
    _lib.check(_lib.lib().kmerlr_select_from_gradient(p(g), nt, N, p(e), p(np.zeros(1)), 0, K.TIE_GO118, 0.0, 0.0,
                                                       p(mask), lam, c, okc))
    o = oracle.select_from_gradient(g, N, [], [], tie=oracle.TIE_GO118)
    assert np.array_equal(mask.astype(bool), o["mask"]) and lam.value == o["lam"] and bool(okc.value) == o["ok"]
    assert c.value == o["c"]
    vals, _ = oracle.nlargest_abs(g[1:], oracle.TIE_GO118)
    assert np.sum(np.abs(g[1:]) == abs(vals[N - 1])) > 2 * N


# ---------------------------------------------------------------------------------------------------
# 9. fold subsets
# ---------------------------------------------------------------------------------------------------
def test_pair_gradient_of_fold_subset(K, c4):
    """subset(train rows) of the whole extraction and from_csr of the same rows: same rows in the same order, the
    same w and the same sums"""
    buf, off, y = c4["seqs"]
    full = K.compile_test_data(None, K.NewKmerCounter(1, 6, revcomp=True), None, None, True, False, (buf, off))
    try:
        full.SetLabels(y)
        sub = full.subset(c4["tr"])
        try:
            rs = sub.rows()
            assert sub.m == 2772 and all(np.array_equal(a, b) for a, b in zip(rs, c4["rows"]["counts"]))
            theta = pair_theta(2772, True, 300, np.random.default_rng(13))
            lr = K.logisticRegression(theta, CW, 0.0, Cooccurrence=True)
            g = lr.Gradient(None, sub)
            assert np.array_equal(g, lr.Gradient(None, c4["f64"]))
            assert np.array_equal(g, lr.Gradient(None, c4["counts"]))
        finally:
            sub.free()
    finally:
        full.free()
