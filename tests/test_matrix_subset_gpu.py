"""kmerlr_matrix_subset (KmerDataSet.subset) and crossvalidation on it: every subset is exactly the numpy selection of
the parent's rows with the parent's columns, gives the same bits on every view (matrix-free, stored rows, an import of
the selected rows, a re-extraction of them against the parent's class list), carries the leapfrog path, the transform
fit and the solvers, outlives its parent, and is refused where it must be.  Needs a B200.

Which bits agree: the stored-row pass of a subset against from_csr of the same rows, and the matrix-free pass of a
subset against the matrix-free pass of a re-extraction of the same rows, add the same row sums in the same order into
fixed-point accumulators: gradient and loss agree bit for bit at every theta.  The matrix-free and the stored-row pass
round differently (a row's weight once per occurrence against once per stored count, and a row's terms added in other
orders), so those two are held to the parity bars both passes meet against the CPU oracle: 1e-10 of max |g| and 1e-12
of the loss."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def sample(K, n_short, n_long, L_short, L_long, M, N, binarize):
    """fg || bg with a few long rows (in both classes) among short ones: the parent's longest row is long"""
    from kmerlr_b200 import synth
    half = n_short // 2
    bs, os_, ys = synth.training_set(half, n_short - half, L_short)
    bl, ol, yl = synth.training_set(n_long // 2, n_long - n_long // 2, L_long, first_fg=10 ** 6, first_bg=10 ** 6)
    buf = np.concatenate([bs, bl])
    off = np.concatenate([os_, ol[1:] + os_[-1]])
    y = np.concatenate([ys, yl])
    kc = K.NewKmerCounter(M, N, revcomp=True, binarize=binarize)
    d = K.compile_test_data(None, kc, None, None, True, binarize, (buf, off))
    d.SetLabels(y)
    return d, kc, buf, off, y


def take(buf, off, rows):
    lens = np.diff(off)
    o = np.concatenate([[0], np.cumsum(lens[rows])]).astype(np.int64)
    b = np.concatenate([buf[off[i]:off[i + 1]] for i in rows])
    return b, o


def select_rows(rp, col, val, idx):
    """numpy selection of CSR rows"""
    lens = np.diff(rp)[idx]
    orp = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    pos = np.concatenate([np.arange(rp[i], rp[i + 1]) for i in idx]) if orp[-1] else np.zeros(0, dtype=np.int64)
    return orp, col[pos], val[pos]


def index_lists(n, rng):
    perm = rng.permutation(n)
    return {"sorted": np.sort(perm[: (4 * n) // 5]), "shuffled": perm[: n // 2], "reversed": np.arange(n)[::-1].copy(),
            "repeated": rng.integers(0, n, size=n), "single": np.array([n - 1]), "every": np.arange(n)}


def grad_loss(K, d, theta, cw):
    lr = K.logisticRegression(theta, cw, 0.0)
    return lr.Gradient(None, d), lr.Loss(d)


# ---------------------------------------------------------------------------------------------------
# 1. rows and numbering
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", ["c2_counts", "c3_binarized"])
def test_rows_and_numbering(K, shape):
    """sorted, shuffled, reversed and repeated index lists, one row and every row, from a padded parent (straight from
    the extraction) and from its compact form: rows, n_global, labels (class weights) and the class list are the numpy
    selection of the parent's"""
    if shape == "c2_counts":
        d, kc, buf, off, y = sample(K, 1500, 20, 500, 1900, 1, 8, False)
    else:
        d, kc, buf, off, y = sample(K, 1500, 20, 200, 1000, 1, 10, True)
    rng = np.random.default_rng(11)
    lists = index_lists(d.n, rng)
    kmers = d.Kmers()
    try:
        subs = {name: d.subset(idx) for name, idx in lists.items()}        # from the padded rows
        rp, col, val = d.rows()                                              # (compacts the parent in place)
        subs.update({name + "/compact": d.subset(idx) for name, idx in lists.items()})
        for name, s in subs.items():
            idx = lists[name.split("/")[0]]
            assert (s.n, s.m, s.n_classes, s.n_global) == (len(idx), d.m, d.n_classes, len(idx)), name
            erp, ecol, evl = select_rows(rp, col, val, idx)
            srp, scol, sval = s.rows()
            assert s.nnz == erp[-1] and np.array_equal(srp, erp) and np.array_equal(scol, ecol) and np.array_equal(sval, evl), name
            k, c = s.Kmers()
            assert np.array_equal(k, kmers[0]) and np.array_equal(c, kmers[1]), name
            assert np.array_equal(s.Labels, y[idx].astype(bool)), name
            if 0 < y[idx].sum() < len(idx):
                assert np.array_equal(s.class_weights(), K.compute_class_weights(y[idx])), name
        for s in subs.values():
            s.free()
    finally:
        d.free()


def test_class_only_in_held_out_rows_keeps_its_column(K):
    """a fold whose held-out rows hold every occurrence of some classes: the training subset keeps those columns (m, the
    class list and the pair coefficient space are the parent's) and their gradient is exactly 0; a re-extraction of the
    training rows would have lost them"""
    d, kc, buf, off, y = sample(K, 400, 0, 60, 60, 1, 6, False)
    try:
        rp, col, val = d.rows()
        counts = np.bincount(col, minlength=d.m)
        rare = np.nonzero(counts == 1)[0][:20]
        assert len(rare) >= 5
        rows_of_rare = np.unique(np.searchsorted(rp, np.nonzero(np.isin(col, rare))[0], side="right") - 1)
        fold = np.arange(d.n) % 5
        fold[rows_of_rare] = 0
        train = d.subset(np.nonzero(fold != 0)[0])
        theta = np.random.default_rng(3).normal(scale=0.05, size=d.m + 1)
        g, _ = grad_loss(K, train, theta, (1.0, 1.0))
        assert train.m == d.m and np.all(g[rare + 1] == 0.0) and np.any(g[1:] != 0.0)
        re = K.compile_test_data(None, kc, None, None, True, False, take(buf, off, np.nonzero(fold != 0)[0]))
        assert re.m < d.m
        re.free(); train.free()
    finally:
        d.free()


# ---------------------------------------------------------------------------------------------------
# 2. the same bits on every view
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("binarize", [False, True])
def test_same_bits_on_every_view(K, binarize):
    """count (k = 1..8) and binarized (k = 1..10) rows; a 4/5 fold, a shuffled half with repeats, and the short rows only
    (a longest row shorter than the parent's: another instantiation of the matrix-free pass); class weights (1, 1) and
    (0.8, 1.3); theta = 0 and a random sparse theta"""
    if binarize:
        d, kc, buf, off, y = sample(K, 1500, 20, 200, 1000, 1, 10, True)
    else:
        d, kc, buf, off, y = sample(K, 1500, 20, 500, 1900, 1, 8, False)
    rng = np.random.default_rng(5)
    perm = rng.permutation(d.n)
    lists = [np.sort(perm[: (4 * d.n) // 5]), np.concatenate([perm[: d.n // 2], perm[:50]]), np.arange(1500)]
    kmers = d.Kmers()
    subs = [d.subset(idx) for idx in lists]
    rp, col, val = d.rows()
    try:
        for idx, s in zip(lists, subs):
            erp, ecol, evl = select_rows(rp, col, val, idx)
            imp = K.from_csr(len(idx), d.m, erp, ecol, evl)
            imp.SetLabels(y[idx])
            ext = K.compile_test_data(None, kc, kmers, None, True, binarize, take(buf, off, idx))
            ext.SetLabels(y[idx])
            assert ext.m == d.m
            theta_r = rng.normal(scale=0.02, size=d.m + 1)
            theta_r[rng.random(d.m + 1) < 0.7] = 0.0
            for theta in (np.zeros(d.m + 1), theta_r):
                for cw in ((1.0, 1.0), (0.8, 1.3)):
                    K.option("implicit", 1)
                    try:
                        g_mf, l_mf = grad_loss(K, s, theta, cw)
                        g_ext, l_ext = grad_loss(K, ext, theta, cw)
                        K.option("implicit", 0)
                        g_st, l_st = grad_loss(K, s, theta, cw)
                    finally:
                        K.option("implicit", 1)
                    g_csr, l_csr = grad_loss(K, imp, theta, cw)
                    assert np.array_equal(g_mf, g_ext) and l_mf == l_ext
                    assert np.array_equal(g_st, g_csr) and l_st == l_csr
                    rel = np.max(np.abs(g_mf - g_st)) / np.max(np.abs(g_st))
                    assert rel <= 1e-10, rel
                    assert abs(l_mf - l_st) <= 1e-12 * abs(l_st)
            imp.free(); ext.free()
    finally:
        for s in subs:
            s.free()
        d.free()


# ---------------------------------------------------------------------------------------------------
# 3. the leapfrog path on a fold
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tie", ["go118", "index"])
def test_leapfrog_path_on_a_fold(K, oracle, tie):
    """a C2-shaped sample (k = 1..8 revcomp), the training rows of fold 0 of 5: the path over --lambda-auto=5,10 on the
    stored rows of the subset equals the path on from_csr of the same rows bit for bit (lambdas, iterations, selected
    sets, theta), the matrix-free subset equals a re-extraction of the rows against the parent's class list bit for bit,
    and both agree with the CPU oracle on those rows to the parity bars of the fixture path test"""
    from kmerlr_b200 import synth
    O = oracle
    buf, off, y = synth.training_set(1000, 1000, 500)
    kc, oc = K.NewKmerCounter(1, 8, revcomp=True), O.make_config(1, 8, revcomp=True)
    d = K.compile_test_data(None, kc, None, None, True, False, (buf, off))
    d.SetLabels(y)
    tr = np.nonzero(np.arange(d.n) % 5 != 0)[0]
    kmers = d.Kmers()
    s = d.subset(tr)
    rp, col, val = d.rows()
    imp = K.from_csr(len(tr), d.m, *select_rows(rp, col, val, tr))
    imp.SetLabels(y[tr])
    ext = K.compile_test_data(None, kc, kmers, None, True, False, take(buf, off, tr))
    ext.SetLabels(y[tr])
    ref = O.extract(oc, take(buf, off, tr), frozen=kmers)
    assert ref.m == d.m
    kt, ot = (K.TIE_GO118, O.TIE_GO118) if tie == "go118" else (K.TIE_INDEX, O.TIE_INDEX)
    try:
        def path(data, implicit):
            K.option("implicit", implicit)
            try:
                est = K.KmerLrEstimator(EpsilonLoss=1e-8, tie=kt, MaxIterations=20000)
                out = []
                for N in (5, 10):
                    est.path = []
                    est.estimate_loop(data, N)
                    out.append((list(est.path), est.active_idx.copy(), est.Theta.copy()))
                return out
            finally:
                K.option("implicit", 1)

        def same(a, b):
            for (pa, ia, ta), (pb, ib, tb) in zip(a, b):
                assert pa == pb and np.array_equal(ia, ib) and np.array_equal(ta, tb)

        stored, mf = path(s, 0), path(s, 1)
        same(stored, path(imp, 1))
        same(mf, path(ext, 1))
        oest = O.EstimatorState()
        for N, (p, idx, theta) in zip((5, 10), mf):
            res = O.estimate_loop(ref, y[tr], (1, 1), N, oest, tie=ot, epsilon_loss=1e-8, max_iter=20000)
            assert len(p) == res["epochs"] and np.array_equal(idx, oest.active_idx)
            assert np.allclose([q[0] for q in p], res["lambdas"], rtol=1e-9, atol=0)
            assert np.max(np.abs(theta - oest.active_theta)) <= 1e-5 * max(1.0, np.max(np.abs(oest.active_theta)))
        # once with the accelerated solver: the subset's stored rows against the import
        runs = []
        for data in (s, imp):
            K.option("implicit", 0)
            try:
                est = K.KmerLrEstimator(EpsilonLoss=1e-8, tie=kt, MaxIterations=20000, Accelerated=True)
                est.estimate_loop(data, 5)
            finally:
                K.option("implicit", 1)
            runs.append((list(est.path), est.active_idx.copy(), est.Theta.copy()))
        same([runs[0]], [runs[1]])
    finally:
        s.free(); imp.free(); ext.free(); d.free()


# ---------------------------------------------------------------------------------------------------
# 4. the transform fit on a fold
# ---------------------------------------------------------------------------------------------------
def test_transform_fit_on_a_fold(K):
    """TransformFull.Fit on a training subset (single and pair moments) equals the fit on a re-extraction of the same rows
    against the parent's class list, and the column sums equal numpy's on the selected rows"""
    d, kc, buf, off, y = sample(K, 600, 10, 300, 900, 1, 4, False)
    tr = np.nonzero(np.arange(d.n) % 5 != 2)[0]
    s = d.subset(tr)
    ext = K.compile_test_data(None, kc, d.Kmers(), None, True, False, take(buf, off, tr))
    rp, col, val = d.rows()
    try:
        for kind in ("standardizer", "max-abs-scaler", "mean-scaler"):
            for cooc in (False, True):
                a = K.TransformFull().Fit(s, kind, cooc)
                b = K.TransformFull().Fit(ext, kind, cooc)
                for x, z in ((a.Offset, b.Offset), (a.Scale, b.Scale)):
                    assert (x is None) == (z is None) and (x is None or np.array_equal(x, z)), (kind, cooc)
        _, ecol, evl = select_rows(rp, col, val, tr)
        m = d.m
        s1, s2, mx = np.zeros(m), np.zeros(m), np.zeros(m)
        cnt = np.zeros(m, dtype=np.int64)
        from kmerlr_b200 import _lib
        _lib.check(_lib.lib().kmerlr_column_moments(s.h, _p(s1), _p(s2), _p(mx), _p(cnt)))
        assert np.array_equal(s1, np.bincount(ecol, weights=evl, minlength=m))
        assert np.array_equal(cnt, np.bincount(ecol, minlength=m))
    finally:
        s.free(); ext.free(); d.free()


# ---------------------------------------------------------------------------------------------------
# 5. lifetime, subsets of subsets, subsets of reduced / imported / transformed matrices
# ---------------------------------------------------------------------------------------------------
def test_lifetime_and_nesting(K):
    """a subset outlives its parent (gradient and a leapfrog epoch after the free equal those before); a subset of a
    subset equals the subset of the composed indices; subsets of a reduced, an imported and a transformed (f64) matrix
    are the numpy selections of their rows with the same bits as from_csr of those rows"""
    for binarize in (False, True):
        d, kc, buf, off, y = sample(K, 800, 8, 200, 700, 1, 8 if not binarize else 10, binarize)
        rng = np.random.default_rng(17)
        a = rng.permutation(d.n)[:600]
        b = np.concatenate([rng.permutation(600)[:400], [0, 0, 599]])
        s = d.subset(a)
        ss = s.subset(b)
        direct = d.subset(a[b])
        theta = rng.normal(scale=0.02, size=d.m + 1)
        theta[rng.random(d.m + 1) < 0.5] = 0.0
        cw = (0.9, 1.1)
        g0, l0 = grad_loss(K, s, theta, cw)
        est0 = K.KmerLrEstimator(EpsilonLoss=1e-8, MaxIterations=5000, MaxEpochs=1, tie=K.TIE_INDEX)
        est0.estimate_loop(s, 5)
        d.free()
        g1, l1 = grad_loss(K, s, theta, cw)
        est1 = K.KmerLrEstimator(EpsilonLoss=1e-8, MaxIterations=5000, MaxEpochs=1, tie=K.TIE_INDEX)
        est1.estimate_loop(s, 5)
        assert np.array_equal(g0, g1) and l0 == l1
        assert est0.path == est1.path and np.array_equal(est0.Theta, est1.Theta)
        gs, ls = grad_loss(K, ss, theta, cw)
        gd, ld = grad_loss(K, direct, theta, cw)
        assert np.array_equal(gs, gd) and ls == ld
        for x, z in zip(ss.rows(), direct.rows()):
            assert np.array_equal(x, z)
        ss.free(); direct.free()
        # reduced, imported and transformed parents
        red = K.select_data(s, np.array([0, 1, 3, 7, 20, 100, s.m], dtype=np.int64))
        red.SetLabels(s.Labels.astype(np.uint8))
        srp, scol, sval = s.rows()
        imported = K.from_csr(s.n, s.m, srp, scol, sval)
        imported.SetLabels(s.Labels.astype(np.uint8))
        tf = K.Transform(Scale=np.concatenate([[1.0], 1.0 / (1.0 + np.arange(red.m) % 3)])).Apply(red)
        tf.SetLabels(s.Labels.astype(np.uint8))
        idx = np.concatenate([rng.permutation(s.n)[:300], [5, 5]])
        for parent in (red, imported, tf):
            sub = parent.subset(idx)
            prp, pcol, pval = parent.rows()
            erp, ecol, evl = select_rows(prp, pcol, pval, idx)
            for x, z in zip(sub.rows(), (erp, ecol, evl)):
                assert np.array_equal(x, z)
            ref = K.from_csr(len(idx), parent.m, erp, ecol, evl)
            ref.SetLabels(s.Labels[idx].astype(np.uint8))
            t = rng.normal(scale=0.05, size=parent.m + 1)
            ga, la = grad_loss(K, sub, t, cw)
            gb, lb = grad_loss(K, ref, t, cw)
            assert np.array_equal(ga, gb) and la == lb
            est = [K.KmerLrEstimator(EpsilonLoss=1e-8, MaxIterations=300) for _ in range(2)]
            for e, x in zip(est, (sub, ref)):
                e.Theta = np.zeros(parent.m + 1)
                e.estimate_proximal(x, 1e-3)
            assert np.array_equal(est[0].Theta, est[1].Theta)
            sub.free(); ref.free()
        red.free(); imported.free(); tf.free(); s.free()


# ---------------------------------------------------------------------------------------------------
# 6. refusals
# ---------------------------------------------------------------------------------------------------
def test_refusals(K):
    """KMERLR_ERR_ARG with a message: an empty list, an index of -1 and of n, a null rows or out pointer.  (A sharded
    matrix is refused too; a single-rank process cannot build one, so that refusal is not exercised here.)"""
    from kmerlr_b200 import _lib
    L = _lib.lib()
    d, _, _, _, _ = sample(K, 100, 0, 100, 100, 1, 4, False)
    try:
        for rows, match in ((np.zeros(0, dtype=np.int64), "at least 1"), (np.array([0, -1]), "row index -1"),
                            (np.array([d.n]), "row index %d" % d.n)):
            with pytest.raises(K.KmerLrError) as e:
                d.subset(rows)
            assert e.value.code == _lib.ERR_ARG and match in str(e.value), str(e.value)
        rows, h = np.array([0, 1], dtype=np.int64), C.c_uint64()
        assert L.kmerlr_matrix_subset(d.h, None, 2, h) == _lib.ERR_ARG and b"null argument" in L.kmerlr_last_error()
        assert L.kmerlr_matrix_subset(d.h, _p(rows), 2, None) == _lib.ERR_ARG and b"null argument" in L.kmerlr_last_error()
    finally:
        d.free()


# ---------------------------------------------------------------------------------------------------
# 7. cross-validation
# ---------------------------------------------------------------------------------------------------
def test_crossvalidation_equals_the_hand_written_loop(K):
    """5 folds (fold = i mod 5) on a C4-shaped sample (pair features, k = 1..6 revcomp), --lambda-auto=3,6: the models
    and held-out predictions of crossvalidation equal a loop over subset + Estimate + SelectData + LogPdf / Loss, and
    every row is predicted exactly once, by the model that did not see it"""
    from kmerlr_b200 import synth
    buf, off, y = synth.training_set(500, 500, 500)
    d = K.compile_test_data(None, K.NewKmerCounter(1, 6, revcomp=True), None, None, True, False, (buf, off))
    d.SetLabels(y)
    fold = K.cv_groups(d.n, 5)
    lam = [3, 6]

    def make():
        return K.KmerLrEstimator(Cooccurrence=True, EpsilonLoss=1e-8, MaxIterations=20000, MaxEpochs=3, tie=K.TIE_INDEX)
    try:
        cv = K.crossvalidation(d, fold, make, lam)
        assert list(cv.Folds) == list(range(5))
        seen = np.zeros(d.n, dtype=np.int64)
        for f in range(5):
            tr, te = np.nonzero(fold != f)[0], np.nonzero(fold == f)[0]
            seen[te] += 1
            train, test = d.subset(tr), d.subset(te)
            est = make()
            for j, n in enumerate(lam):
                est.Estimate(train, [n])
                ai, th, tf = cv.Models[f][j]
                assert np.array_equal(ai, est.active_idx) and np.array_equal(th, est.Theta) and tf is None
                sel = K.select_data(test, np.concatenate([[0], est.active_idx]))
                lr = K.logisticRegression(est.Theta, est.ClassWeights, 0.0)
                assert np.array_equal(cv.Predictions[j][te], lr.LogPdf(sel))
                assert cv.Loss[f][j] == lr.Loss(sel)
                sel.free()
            train.free(); test.free()
        assert np.all(seen == 1)
        assert all(np.all(p < 0.0) for p in cv.Predictions)
    finally:
        d.free()


def test_crossvalidation_with_a_transform_and_class_weights(K):
    """3 folds given as explicit, shuffled fold ids, a standardizer fitted on every training subset and balanced class
    weights (--lambda-auto=2,4): the same as the hand-written loop, transforms included"""
    d, kc, buf, off, y = sample(K, 300, 0, 120, 120, 1, 4, False)
    fold = np.random.default_rng(4).permutation(np.arange(d.n) % 3) + 7
    lam = [2, 4]

    def make():
        return K.KmerLrEstimator(EpsilonLoss=1e-8, MaxIterations=20000, tie=K.TIE_GO118)
    try:
        cv = K.crossvalidation(d, fold, make, lam, balance=True, transform_kind="standardizer")
        assert list(cv.Folds) == [7, 8, 9]
        for fi, f in enumerate((7, 8, 9)):
            tr, te = np.nonzero(fold != f)[0], np.nonzero(fold == f)[0]
            train, test = d.subset(tr), d.subset(te)
            t = K.TransformFull().Fit(train, "standardizer")
            est = make()
            for j, n in enumerate(lam):
                est.Estimate(train, [n], True, t)
                ai, th, tf = cv.Models[fi][j]
                assert np.array_equal(ai, est.active_idx) and np.array_equal(th, est.Theta)
                assert np.array_equal(tf.Offset, est.Transform.Offset) and np.array_equal(tf.Scale, est.Transform.Scale)
                sel = K.select_data(test, np.concatenate([[0], est.active_idx]))
                lr = K.logisticRegression(est.Theta, est.ClassWeights, 0.0, False, est.Transform)
                assert np.array_equal(cv.Predictions[j][te], lr.LogPdf(sel)) and cv.Loss[fi][j] == lr.Loss(sel)
                sel.free()
            train.free(); test.free()
    finally:
        d.free()
