"""Generates tests/golden/ref_fixtures.npz from the reference's own test fixtures.

It needs a checkout of the reference (pbenner/kmerLr), which the tests themselves do not:
    python tests/golden/make_fixtures.py <reference checkout>
The fixtures are DATA (FASTA sequences and score tables the reference's tests read,
kmerLr_test.go / scoresLr_test.go), stored as uint8 / float64 arrays.  The golden numbers
those tests assert are transcribed, with file:line, in tests/test_oracle_golden.py.
"""
import os
import sys

import numpy as np

if len(sys.argv) != 2:
    sys.exit(__doc__)
REF = sys.argv[1]
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_fixtures.npz")


def read_fasta(path):
    seqs, cur = [], None
    with open(path) as f:
        for line in f:
            line = line.strip()
            if not line:
                continue
            if line.startswith(">"):
                if cur is not None:
                    seqs.append("".join(cur))
                cur = []
            else:
                cur.append(line)
    if cur is not None:
        seqs.append("".join(cur))
    return seqs


def pack(seqs):
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(s) for s in seqs])
    return np.frombuffer("".join(seqs).encode(), dtype=np.uint8).copy(), off


def read_table(path):
    rows = []
    with open(path) as f:
        for line in f:
            line = line.strip()
            if line:
                rows.append([float(x) for x in line.split(",")])
    return np.array(rows, dtype=np.float64)


out = {}
for name in ("kmerLr_test", "kmerLr_test_fg", "kmerLr_test_bg", "kmerLr_test_co_fg", "kmerLr_test_co_bg"):
    buf, off = pack(read_fasta(os.path.join(REF, name + ".fa")))
    out[name + "_seq"], out[name + "_off"] = buf, off
for name in ("scoresLr_test_fg", "scoresLr_test_bg", "scoresLr_test_co_fg", "scoresLr_test_co_bg"):
    out[name] = read_table(os.path.join(REF, name + ".table"))
np.savez_compressed(OUT, **out)
print("wrote", OUT, {k: v.shape for k, v in out.items()})
