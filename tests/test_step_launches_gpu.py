"""Launch budget of one training step (extract + labels + one proximal-gradient iteration), the numbering set the
extraction keeps per configuration, and the fused tail of the matrix-free pass against the stored-row pass.
Needs a B200."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def sample(n=300, L=400, seed=0):
    from kmerlr_b200 import synth
    return synth.training_set(n, n, L, first_fg=seed * n, first_bg=seed * n)


def rows_of(d):
    rp, col, val = d.rows()
    k, code = d.Kmers()
    return rp, col, val, np.asarray(k), np.asarray(code)


def same(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


def test_step_launch_budget(K):
    """extract: the kernel, its totals and the class list; labels: one kernel; one matrix-free iteration: build
    the tables, the pass, the fold, the pass tail and the prox update, then the loss-only pass and its tail.
    (k <= 6 on 600 rows: every class occurs, as at C2, so no renumbering)"""
    from kmerlr_b200 import api
    buf, off, y = sample()
    counter = K.NewKmerCounter(1, 6, revcomp=True)
    seqs = K.Sequences((buf, off))
    api._extract(counter, seqs, None, None, False).free()      # the configuration's numbering set is built once
    counts = []
    for _ in range(2):
        l0 = K.launch_count()
        d = api._extract(counter, seqs, None, None, False)
        l1 = K.launch_count()
        d.SetLabels(y)
        l2 = K.launch_count()
        est = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=1e-300, MaxIterations=1)
        est.Theta = np.zeros(d.m + 1)
        est.estimate_proximal(d, 1e-3)
        l3 = K.launch_count()
        counts.append((l1 - l0, l2 - l1, l3 - l2))
        d.free()
    seqs.free()
    assert counts[0] == counts[1]
    ext, lab, pg = counts[0]
    assert ext <= 3 and lab <= 1 and pg <= 10, counts
    assert ext + lab + pg <= 15


def test_cached_numbering_set_gives_the_same_matrix(K):
    buf, off, _ = sample(seed=1)
    kc = K.NewKmerCounter(1, 8, revcomp=True)
    a = K.compile_test_data(None, kc, None, None, True, False, (buf, off))
    b = K.compile_test_data(None, kc, None, None, True, False, (buf, off))
    assert same(rows_of(a), rows_of(b))
    a.free(); b.free()


@pytest.mark.parametrize("flags", [dict(reverse=True), dict(complement=True)])
def test_frozen_and_unfrozen_extractions_do_not_share_numbering(K, flags):
    """a frozen class list numbers its own columns; the cached set of every class of the configuration is not
    touched by it, in either order"""
    buf, off, _ = sample(seed=2)
    kc = K.NewKmerCounter(2, 7, **flags)
    free1 = K.compile_test_data(None, kc, None, None, True, False, (buf, off))
    k, code = free1.Kmers()
    sub = (np.asarray(k)[1::3], np.asarray(code)[1::3])
    froz1 = K.compile_test_data(None, kc, sub, None, True, False, (buf, off))
    free2 = K.compile_test_data(None, kc, None, None, True, False, (buf, off))
    froz2 = K.compile_test_data(None, kc, sub, None, True, False, (buf, off))
    assert same(rows_of(free1), rows_of(free2))
    assert same(rows_of(froz1), rows_of(froz2))
    fk, fc = froz1.Kmers()
    assert np.array_equal(np.asarray(fk), sub[0]) and np.array_equal(np.asarray(fc), sub[1])
    assert froz1.m == len(sub[0]) and free1.m > froz1.m
    # a subset of the sequences may miss classes: the columns are renumbered, the cached set stays as it was
    part = K.compile_test_data(None, kc, None, None, True, False, (buf[:off[4]], off[:5]))
    free3 = K.compile_test_data(None, kc, None, None, True, False, (buf, off))
    assert part.m < free1.m and same(rows_of(free1), rows_of(free3))
    for d in (free1, froz1, free2, froz2, part, free3):
        d.free()


def test_matrix_free_iterations_equal_stored_row_iterations(K):
    buf, off, y = sample(seed=3)
    d = K.compile_test_data(None, K.NewKmerCounter(1, 8, revcomp=True), None, None, True, False, (buf, off))
    d.SetLabels(y)
    thetas = []
    for implicit in (1, 0):
        K.option("implicit", implicit)
        try:
            est = K.KmerLrEstimator(Epsilon=0.0, EpsilonLoss=1e-300, MaxIterations=6)
            est.Theta = np.zeros(d.m + 1)
            est.ClassWeights = np.array([0.9, 1.2])
            est.estimate_proximal(d, 1e-3)
            thetas.append((np.array(est.Theta), est.hook_state))
        finally:
            K.option("implicit", 1)
    (t1, h1), (t0, h0) = thetas
    assert np.any(t1[1:] != 0.0)
    assert np.max(np.abs(t1 - t0)) <= 1e-13 * max(np.max(np.abs(t0)), 1e-300)
    assert np.all(np.isfinite(h1)) and np.allclose(h1, h0, rtol=1e-13, atol=0.0)
    d.free()
