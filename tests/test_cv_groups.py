"""CPU checks of the cross-validation bookkeeping: the round-robin fold assignment and the scatter of the held-out
results back to row order."""
import numpy as np
import pytest


def test_cv_groups_is_round_robin():
    """getCvGroups (kmerLr_crossvalidation.go:56) before its shuffle: row i goes to fold i mod k"""
    import kmerlr_b200 as K
    for n, k in ((0, 3), (1, 1), (7, 3), (20000, 5), (4, 9)):
        g = K.cv_groups(n, k)
        assert g.dtype == np.int64 and np.array_equal(g, np.array([i % k for i in range(n)], dtype=np.int64))
        assert np.array_equal(np.bincount(g, minlength=k)[:min(n, k)], [len(range(f, n, k)) for f in range(min(n, k))])
    with pytest.raises(K.KmerLrError):
        K.cv_groups(5, 0)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_held_out_results_go_back_to_their_rows(seed):
    """fold ids in any order (shuffled, gaps between the ids): fold f's held-out values, listed in ascending row order,
    land at exactly the rows of fold f, and every row is written once"""
    import kmerlr_b200 as K
    rng = np.random.default_rng(seed)
    n = 1000
    ids = rng.permutation(np.arange(n) % 5) * 3 + 2           # fold ids 2, 5, 8, 11, 14
    value = rng.normal(size=n)
    held_out = [value[np.nonzero(ids == f)[0]] for f in np.unique(ids)]
    out = K.cv_scatter(ids, held_out)
    assert np.array_equal(out, value)
    marks = K.cv_scatter(ids, [np.ones(len(h)) for h in held_out])
    assert np.array_equal(marks, np.ones(n))
