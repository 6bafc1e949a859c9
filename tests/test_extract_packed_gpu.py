"""Revcomp configurations with N <= 8 sort their sorted level on 16-bit keys, two to a register, with 0xFFFF
as the sentinel.  Parity with the CPU oracle at every keys-per-lane width (E = 2 .. 64), with rows full of the
extreme codes (AAAAAAAA, TTTTTTTT: the sentinel's bit pattern), long runs of one key across lanes, invalid
bases, counts and binarized rows, and a frozen class list.  Needs a B200."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def rows_for(rng, L, n):
    seqs = []
    for i in range(n):
        kind = i % 5
        if kind == 0:
            s = rng.choice(list("ACGT"), size=L)
        elif kind == 1:
            s = np.array(list(("T" * 40 + "A" * 40) * (L // 80 + 1))[:L])     # codes 0xFFFF and 0 in long runs
        elif kind == 2:
            s = rng.choice(list("AT"), size=L)                                  # few classes, long runs
        elif kind == 3:
            s = np.array(list("T" * L))                                         # one class: TTTTTTTT = AAAAAAAA
        else:
            s = rng.choice(list("ACGTN"), size=L)                               # invalid bases cut the windows
        seqs.append("".join(s))
    return seqs


@pytest.mark.parametrize("L", [50, 100, 250, 500, 1000, 2000])
@pytest.mark.parametrize("M,N,binz", [(1, 8, False), (8, 8, False), (1, 8, True), (4, 8, True)])
def test_packed_sort_parity(K, oracle, L, M, N, binz):
    rng = np.random.default_rng(L * 31 + M * 7 + N + binz)
    seqs = rows_for(rng, L, 25) + rows_for(rng, int(rng.integers(0, L + 1)), 5)
    kc, oc = K.NewKmerCounter(M, N, revcomp=True, binarize=binz), oracle.make_config(M, N, revcomp=True, binarize=binz)
    d = K.compile_test_data(None, kc, None, None, True, binz, seqs)
    ref = oracle.extract(oc, seqs)
    assert (d.n, d.m, d.nnz) == (ref.n, ref.m, ref.nnz)
    k, c = d.Kmers()
    rk, rc = ref.classes()
    assert np.array_equal(k, rk) and np.array_equal(c, rc)
    for x, y in zip(d.rows(), ref.rows()):
        assert np.array_equal(x, y)
    sub = (k[::2], c[::2])                                                      # frozen list: every other class
    ds = K.compile_test_data(None, kc, sub, None, True, binz, seqs)
    rs = oracle.extract(oc, seqs, frozen=sub)
    assert (ds.n, ds.m, ds.nnz) == (rs.n, rs.m, rs.nnz)
    for x, y in zip(ds.rows(), rs.rows()):
        assert np.array_equal(x, y)
