"""FASTA text parsed on the device (import_fasta) and regions cut out of a resident set (Sequences.regions) against
the existing host path: the same sets base for base, the same matrices, labels, scores and wiggle bytes."""
import ctypes as C

import numpy as np
import pytest

from conftest import cat
from fasta_rule import LAYOUTS, fixture_sets, layout_text, letters, read_fasta


def check_same_set(K, texts):
    """import_fasta(*texts) against Sequences(read_fasta(text) of every text): names, records, lengths, bases"""
    s = K.import_fasta(*texts)
    names, seqs, records = [], [], []
    for t in texts:
        a, b = read_fasta(t)
        names += a
        seqs += b
        records.append(len(a))
    assert s.records == records
    assert [x.encode("utf-8", "surrogateescape") for x in s.names] == names
    assert s.n == len(seqs) and s.total_bases == sum(len(x) for x in seqs)
    assert s.lengths().tolist() == [len(x) for x in seqs]
    got = s.bases()
    assert got == letters(b"".join(seqs))
    ref = K.Sequences(seqs)
    assert ref.bases() == got
    return s


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS, ids=[str(i) for i in range(len(LAYOUTS))])
def test_fixture_layouts(K, fixtures, layout):
    texts = []
    for name, seqs in fixture_sets(fixtures):
        names = [b"%s_%d description" % (name.encode(), i) for i in range(len(seqs))]
        texts.append(layout_text(names, seqs, layout)[0])
    for t in texts:
        check_same_set(K, [t])
    check_same_set(K, texts)


@pytest.mark.gpu
def test_awkward_texts(K):
    rng = np.random.default_rng(5)
    iupac = b"ACGTNRYKMSWBDHVacgtnrykmswbdhv-.*"
    high = bytes(range(0x80, 0x100))
    texts = [
        b"", b"\n\n  \r\n", b">", b">\n>\n>", b">only\n>headers\n",
        b">n runs\n" + b"N" * 1000 + b"\nACGT" + b"n" * 77 + b"\n" + b"NNNNACGT" * 40 + b"\n",
        b">iupac\n" + bytes(rng.choice(np.frombuffer(iupac, dtype=np.uint8), 5000)) + b"\n",
        b">high \xff\xfe name\n" + bytes(rng.choice(np.frombuffer(high + b"ACGT", dtype=np.uint8), 3000)) + b"\n",
        b">lower\nacgtacgtnnacgt\n>inner spaces\nAC GT\tAC  GT\r\n  AC GT  \n",
        b">  \t\n" + b"ACGT" * 50 + b"\n>\nAC\n",
        b">last line without newline\nACGTACGT\nAC",
        b">a\rb\nAC\rGT\rAC\n",
    ]
    for t in texts:
        check_same_set(K, [t])
    check_same_set(K, texts)


@pytest.mark.gpu
def test_one_long_line(K):
    rng = np.random.default_rng(6)
    seq = np.frombuffer(b"ACGTacgtN", dtype=np.uint8)[rng.integers(0, 9, 250_000_000)].tobytes()
    text = b">chrL long contig\n" + seq + b"\n>short\nACGT\n"
    s = K.import_fasta(text)
    assert s.names == ["chrL long contig", "short"] and s.lengths().tolist() == [250_000_000, 4]
    assert s.bases() == letters(seq) + b"acgt"


@pytest.mark.gpu
def test_many_records(K):
    rng = np.random.default_rng(7)
    n = 200_000
    lens = rng.integers(0, 300, n)
    pool = np.frombuffer(b"ACGTN", dtype=np.uint8)[rng.integers(0, 5, int(lens.sum()))].tobytes()
    off = np.concatenate([[0], np.cumsum(lens)])
    seqs = [pool[off[i]:off[i + 1]] for i in range(n)]
    names = [b"rec%d" % i for i in range(n)]
    check_same_set(K, [layout_text(names[:n // 2], seqs[:n // 2], dict(width=80))[0],
                       layout_text(names[n // 2:], seqs[n // 2:], dict(width=61, eol=b"\r\n"))[0]])


@pytest.mark.gpu
def test_text_above_2_31_bytes(K):
    """one text of more than 2^31 bytes: lengths, names and regions cut out beyond the 2^31st byte"""
    rng = np.random.default_rng(8)
    line = np.frombuffer(b"ACGTN", dtype=np.uint8)[rng.integers(0, 5, 60)]
    reps = (1 << 31) // 61 + 1000
    head, tail = b">big\n", b">tail record\nACGTTGCA\n"
    text = np.empty(len(head) + 61 * reps + len(tail), dtype=np.uint8)
    text[:len(head)] = np.frombuffer(head, dtype=np.uint8)
    body = text[len(head):len(head) + 61 * reps].reshape(reps, 61)
    body[:, :60] = line
    body[:, 60] = ord("\n")
    text[len(head) + 61 * reps:] = np.frombuffer(tail, dtype=np.uint8)
    assert len(text) > (1 << 31)
    s = K.import_fasta(text)
    del text, body
    L = 60 * reps
    assert s.names == ["big", "tail record"] and s.lengths().tolist() == [L, 8] and s.records == [2]
    cross = ((1 << 31) - len(head)) * 60 // 61          # the base whose byte in the text is near byte 2^31
    starts = [0, cross - 37, L - 1000, L - 64, L - 1]
    r = s.regions([0] * len(starts) + [1], starts + [0], [a + min(1000, L - a) for a in starts] + [8])
    want = b"".join(letters(line[np.arange(a, a + min(1000, L - a)) % 60].tobytes()) for a in starts) + b"acgttgca"
    assert r.bases() == want


def training_pair(fixtures, fg, bg, layout):
    out = []
    for name in (fg, bg):
        buf, off = fixtures[name + "_seq"], fixtures[name + "_off"]
        seqs = [buf[off[i]:off[i + 1]].tobytes() for i in range(len(off) - 1)]
        out.append(layout_text([b"%d" % i for i in range(len(seqs))], seqs, layout)[0])
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("fg,bg,M,N,flags", [
    ("kmerLr_test_fg", "kmerLr_test_bg", 1, 6, dict(revcomp=True)),                          # C1
    ("kmerLr_test_co_fg", "kmerLr_test_co_bg", 2, 6, dict(revcomp=True, binarize=True)),     # TestKmers6's data
    ("kmerLr_test_fg", "kmerLr_test_bg", 4, 8, dict(revcomp=True, alphabet="gapped-nucleotide")),
])
def test_same_matrices(K, fixtures, fg, bg, M, N, flags):
    buf, off, labels = cat(fixtures, fg, bg)
    flags = dict(flags)
    binarize = flags.pop("binarize", False)
    kc = K.NewKmerCounter(M, N, **flags)
    nfg = len(fixtures[fg + "_off"]) - 1
    ref = K.compile_training_data(None, kc, None, None, True, binarize, (buf[:off[nfg]], off[:nfg + 1]),
                                  (buf[off[nfg]:], off[nfg:] - off[nfg]))
    theta = np.linspace(-0.02, 0.03, ref.m + 1)
    g_ref = K.logisticRegression(theta).Gradient(None, ref)
    for layout in (dict(width=60), dict(width=7, eol=b"\r\n", blank=True)):
        s = K.import_fasta(*training_pair(fixtures, fg, bg, layout))
        d = K.compile_training_data(None, kc, None, None, True, binarize, s)
        assert np.array_equal(d.Labels, labels.astype(bool)) and np.array_equal(d.Labels, ref.Labels)
        for a, b in zip(d.Kmers(), ref.Kmers()):
            assert np.array_equal(a, b)
        for a, b in zip(d.rows(), ref.rows()):
            assert np.array_equal(a, b)
        g = K.logisticRegression(theta).Gradient(None, d)
        assert np.array_equal(g, g_ref)
        # compile_test_data / compile_data on the same resident set
        t = K.compile_test_data(None, kc, ref.Kmers(), None, True, binarize, s)
        for a, b in zip(t.rows(), ref.rows()):
            assert np.array_equal(a, b)
        sets = K.compile_data(None, kc, None, None, True, binarize, s)
        want = K.compile_data(None, kc, None, None, True, binarize,
                              [(buf[:off[nfg]], off[:nfg + 1]), (buf[off[nfg]:], off[nfg:] - off[nfg])])
        for x, y in zip(sets, want):
            for a, b in zip(x.rows(), y.rows()):
                assert np.array_equal(a, b)


def genome(rng, lens):
    seqs = [np.frombuffer(b"ACGTacgtN", dtype=np.uint8)[rng.integers(0, 9, n)].tobytes() for n in lens]
    return [b"chr%d" % (i + 1) for i in range(len(lens))], seqs


def random_regions(rng, lens):
    """every start offset modulo 64, empty regions, regions at contig ends, whole contigs"""
    reg = []
    for i, n in enumerate(lens):
        reg += [(i, 0, n), (i, n, n), (i, 0, 0)]
        for a in range(64):
            if a + 64 <= n:
                reg.append((i, a, int(rng.integers(a, min(n, a + 3000) + 1))))
        for _ in range(20):
            a = int(rng.integers(0, n + 1))
            reg += [(i, a, int(rng.integers(a, n + 1))), (i, a, n)]
    return reg


@pytest.mark.gpu
def test_regions(K, tmp_path):
    from kmerlr_b200 import _lib
    rng = np.random.default_rng(9)
    lens = [100_003, 0, 64, 6_400, 50_001, 1]
    names, seqs = genome(rng, lens)
    g = K.import_fasta(layout_text(names, seqs, dict(width=60))[0])
    reg = random_regions(rng, lens)
    idx, frm, to = (np.array(x, dtype=np.int64) for x in zip(*reg))
    r = g.regions(idx, frm, to)
    host = [seqs[i][a:b] for i, a, b in reg]
    assert r.lengths().tolist() == [len(x) for x in host]
    assert r.bases() == letters(b"".join(host)) == K.Sequences(host).bases()
    # scores of the regions against the host path, then the wiggle file from the scores that stay on the device
    kc = K.NewKmerCounter(1, 6, revcomp=True)
    d = K.compile_test_data(None, kc, None, None, True, False, host)
    ck, cc = d.Kmers()
    sel = np.sort(rng.choice(d.m, 40, replace=False))
    model = dict(counter=kc, class_k=ck[sel], class_code=cc[sel], features=[[i, i] for i in range(40)],
                 theta=rng.normal(size=41) * 0.1, summary="")
    gm = K.genomicKmerLr([model])
    W, step = 200, 10
    preds = gm.predict_window_genomic(host, W, step)
    total = sum(len(p) for p in preds)
    res = gm.predict_resident(r, W, step, fetch=True, total_slots=total)
    assert np.array_equal(res[:total], np.concatenate(preds))
    regions = [(names[i].decode(), a) for i, a, b in reg]
    f1 = str(tmp_path / "host.wig")
    K.saveWindowPredictionsWiggle(f1, regions, preds, "t", W, step)
    h = _lib.C.c_uint64(0)
    K.api.check(K.api.lib().kmerlr_score_windows_resident(gm._arr, 1, r.h, W, step, None, C.byref(h)))
    f2 = str(tmp_path / "dev.wig")
    K.saveWindowPredictionsWiggle(f2, regions, [len(p) for p in preds], "t", W, step, scores=h.value)
    K.api.check(K.api.lib().kmerlr_free(h.value))
    assert open(f1, "rb").read() == open(f2, "rb").read()
    # regions of a set made by the existing path, and no regions at all
    assert K.Sequences(seqs).regions(idx, frm, to).bases() == r.bases()
    e = g.regions([], [], [])
    assert e.n == 0 and e.bases() == b""


@pytest.mark.gpu
def test_refusals(K):
    def refused(match, f, *a):
        with pytest.raises(K.KmerLrError, match=match) as e:
            f(*a)
        assert e.value.code == 1

    refused("text 0 has sequence data before its first header", K.import_fasta, b"ACGT\n>a\nAC\n")
    refused("text 1 has sequence data before its first header", K.import_fasta, b">a\nAC\n", b"\n  GT\n>b\n")
    refused("text 1 is gzip-compressed", K.import_fasta, b">a\nAC\n", b"\x1f\x8b\x08\x00\x00")
    s = K.import_fasta(b">a\nACGTACGT\n>b\n\n>c\nAC\n")
    refused("sequence index 3 out of range", s.regions, [3], [0], [1])
    refused("sequence index -1 out of range", s.regions, [-1], [0], [1])
    refused(r"\[-1, 2\) is not a slice of sequence 0", s.regions, [0], [-1], [2])
    refused(r"\[0, 9\) is not a slice of sequence 0", s.regions, [0], [0], [9])
    refused(r"\[5, 4\) is not a slice of sequence 0", s.regions, [0], [5], [4])
    refused(r"\[0, 1\) is not a slice of sequence 1 \(length 0\)", s.regions, [1], [0], [1])
    assert s.regions([1, 2, 0], [0, 2, 8], [0, 2, 8]).lengths().tolist() == [0, 0, 0]
