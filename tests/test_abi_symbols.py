"""CPU checks of the boundary: the C-ABI library loads, exports every symbol include/kmerlr_b200.h
declares, and fails loudly (no fallback) when there is no GPU."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "kmerlr_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(kmerlr_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_agree():
    from kmerlr_b200 import _lib
    assert header_symbols() == sorted(_lib.SYMBOLS)


def test_library_exports_every_declared_symbol():
    from kmerlr_b200 import _lib
    assert os.path.exists(_lib.SO_PATH), "build the library first: python __graft_entry__.py"
    out = subprocess.check_output(["nm", "-D", "--defined-only", _lib.SO_PATH]).decode()
    exported = set(re.findall(r"\bT (kmerlr_[a-z0-9_]+)", out))
    assert set(header_symbols()) <= exported
    L = _lib.lib()
    for s in header_symbols():
        assert hasattr(L, s)
    assert L.kmerlr_version() == 100


def test_library_is_sm100a_only():
    from kmerlr_b200 import _lib
    out = subprocess.check_output(["cuobjdump", "--list-elf", _lib.SO_PATH]).decode()
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}


def test_pure_host_entry_points():
    """CoeffIndex and the slot count are plain arithmetic (kmerLr_coefficients_index.go:26-54,
    kmerLr_predict_genomic.go:152-156) and need no GPU"""
    import kmerlr_b200 as K
    n = 70
    ci = K.CoeffIndex(n)
    assert ci.Dim() == 2486
    seen = []
    for a in range(n):
        for b in range(a, n):
            j = ci.Ind2Sub(a, b)
            assert ci.Sub2Ind(j - 1) == (a, b)
            seen.append(j)
    assert sorted(seen) == list(range(1, ci.Dim()))
    from kmerlr_b200 import _lib
    L = _lib.lib()
    # Sub2Ind decodes a pair index with a floating-point sqrt.  A float64 restatement of that formula is exact at every
    # index up to m = 20 000 and at the row edges up to m ~ 9.5e7; it first fails near m = 2e8, a pair space far
    # larger than fits in device memory.  Every index of C4 (m = 2 772), then the row edges and random indices of
    # m = 65 536 and 10^6.
    import ctypes as C
    import numpy as np
    a_, b_ = C.c_int64(), C.c_int64()
    sub2ind, ind2sub = L.kmerlr_coeff_sub2ind, L.kmerlr_coeff_ind2sub

    def pair_of(m, j):
        sub2ind(m, j - 1, a_, b_)
        return a_.value, b_.value

    m = 2772
    for a in range(m - 1):
        first = ind2sub(m, a, a + 1)
        for b in range(a + 1, m):
            assert pair_of(m, first + b - a - 1) == (a, b)
        assert ind2sub(m, a, m - 1) == first + m - a - 2
    assert ind2sub(m, m - 2, m - 1) == L.kmerlr_coeff_dim(m) - 1 == 3843378
    rng = np.random.default_rng(0)
    for m in (65536, 10 ** 6):
        dim = L.kmerlr_coeff_dim(m)
        assert dim == (m + 1) * m // 2 + 1
        assert pair_of(m, m + 1) == (0, 1) and pair_of(m, dim - 1) == (m - 2, m - 1)
        for a in range(m - 1):
            first = m + m * (m - 1) // 2 - (m - a) * (m - a - 1) // 2 + 1
            assert ind2sub(m, a, a + 1) == first
            assert pair_of(m, first) == (a, a + 1) and pair_of(m, first + m - a - 2) == (a, m - 1)
        for j in rng.integers(m + 1, dim, 20000):
            a, b = pair_of(m, int(j))
            assert 0 <= a < b < m and ind2sub(m, a, b) == j
    assert L.kmerlr_window_slots(300, 200, 10) == 11 and L.kmerlr_window_slots(200, 200, 10) == 0


def test_no_gpu_fails_loudly():
    """the product path has no CPU fallback: without a usable GPU every compute call errors"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import kmerlr_b200 as K
    with pytest.raises(K.KmerLrError) as e:
        K.init(0)
    assert e.value.code == 4
    with pytest.raises(K.KmerLrError):
        K.compile_test_data(None, K.NewKmerCounter(1, 4), None, None, True, False, ["ACGT"])
    with pytest.raises(K.KmerLrError):
        K.from_dense([[1.0, 2.0]])


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "kmerlr_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.lower().replace("no cpu fallback", ""), f
