"""The FASTA rule on the test side: read_fasta restates, in plain Python on bytes, what the device parser of
import_fasta does (DESIGN §4.7); write_fasta serialises sequences the ways real files come.

It is the rule tests/golden/make_fixtures.py:read_fasta used to turn the reference's fixtures into
ref_fixtures.npz, stated on bytes: lines end at b"\\n" only (a lone b"\\r" inside a line is a byte of that line,
unlike Python's universal newlines)."""
import numpy as np

WS = b" \t\r\v\f"


class FastaError(ValueError):
    pass


def read_fasta(text):
    """bytes -> (names, seqs), both lists of bytes"""
    text = bytes(text)
    if text[:2] == b"\x1f\x8b":
        raise FastaError("gzip-compressed text")
    names, seqs = [], []
    for line in text.split(b"\n"):
        line = line.strip(WS)
        if not line:
            continue
        if line[:1] == b">":
            names.append(line[1:].strip(WS))
            seqs.append([])
        elif not seqs:
            raise FastaError("sequence data before the first header")
        else:
            seqs[-1].append(line)
    return names, [b"".join(s) for s in seqs]


def letters(seq):
    """what the read-back of a packed sequence gives: a/c/g/t in lower case, n for every other byte"""
    a = np.frombuffer(bytes(seq), dtype=np.uint8) | 0x20
    ok = (a == ord("a")) | (a == ord("c")) | (a == ord("g")) | (a == ord("t"))
    return np.where(ok, a, ord("n")).astype(np.uint8).tobytes()


def write_fasta(names, seqs, width=None, eol=b"\n", blank=False, trailing=b"", final_eol=True):
    """width: bases per line (None = unwrapped); blank: an empty line after every header and every record;
    trailing: bytes appended to every line (stripped again by the reader)"""
    out = []
    for name, s in zip(names, seqs):
        out.append(b">" + name + trailing)
        if blank:
            out.append(b"")
        step = width or max(len(s), 1)
        out += [s[j:j + step] + trailing for j in range(0, len(s), step)]
        if blank:
            out.append(b"   " if trailing else b"")
    text = eol.join(out)
    return text + eol if final_eol and out else text


def fixture_sets(fixtures):
    """the reference's fixture sets as (name, [bytes]) pairs"""
    for name in ("kmerLr_test", "kmerLr_test_fg", "kmerLr_test_bg", "kmerLr_test_co_fg", "kmerLr_test_co_bg"):
        buf, off = fixtures[name + "_seq"], fixtures[name + "_off"]
        yield name, [buf[off[i]:off[i + 1]].tobytes() for i in range(len(off) - 1)]


# the layouts every fixture set is written in: line widths, LF / CRLF, blank lines, trailing blanks, empty
# records, no final newline
LAYOUTS = [
    dict(width=1), dict(width=7), dict(width=60), dict(width=61), dict(width=80), dict(width=None),
    dict(width=60, eol=b"\r\n"), dict(width=7, eol=b"\r\n", final_eol=False),
    dict(width=61, blank=True), dict(width=80, trailing=b" \t "), dict(width=None, eol=b"\r\n", blank=True,
                                                                          trailing=b"  "),
    dict(width=60, final_eol=False), dict(width=80, empty_records=True), dict(width=1, empty_records=True,
                                                                             eol=b"\r\n", final_eol=False),
]


def layout_text(names, seqs, layout):
    """(text, expected names, expected seqs) of one layout; empty_records puts an empty record before every other
    record and one at the end"""
    layout = dict(layout)
    if layout.pop("empty_records", False):
        n2, s2 = [], []
        for i, (a, b) in enumerate(zip(names, seqs)):
            if i % 2 == 0:
                n2.append(b"empty%d" % i)
                s2.append(b"")
            n2.append(a)
            s2.append(b)
        names, seqs = n2 + [b"last empty"], s2 + [b""]
    return write_fasta(names, seqs, **layout), names, seqs
