"""CPU checks of the FASTA rule (tests/fasta_rule.py): the reference's fixtures, written out as FASTA in the layouts
real files come in, read back to exactly the stored sequences; the two refusals."""
import pytest

from fasta_rule import LAYOUTS, FastaError, fixture_sets, layout_text, letters, read_fasta


@pytest.mark.parametrize("layout", LAYOUTS, ids=[str(i) for i in range(len(LAYOUTS))])
def test_fixtures_round_trip(fixtures, layout):
    for name, seqs in fixture_sets(fixtures):
        names = [b"%s_%d some description" % (name.encode(), i) for i in range(len(seqs))]
        text, want_names, want_seqs = layout_text(names, seqs, layout)
        got_names, got_seqs = read_fasta(text)
        assert got_names == want_names and got_seqs == want_seqs, name


def test_rule_details():
    assert read_fasta(b"") == ([], [])
    assert read_fasta(b"\n \r\n\t\n") == ([], [])
    assert read_fasta(b">") == ([b""], [b""])
    assert read_fasta(b">a\n>b\n") == ([b"a", b"b"], [b"", b""])
    # the whole header is the name; inner bytes of a sequence line are kept
    assert read_fasta(b">  chr1 x y \r\nac gt\r\nNN\n") == ([b"chr1 x y"], [b"ac gtNN"])
    # a lone \r is a byte of its line, not a line break
    assert read_fasta(b">a\rb\nac\rgt") == ([b"a\rb"], [b"ac\rgt"])
    # a line starting with '>' after blanks is a header
    assert read_fasta(b"  >x\nacgt\n") == ([b"x"], [b"acgt"])
    assert letters(b"AcGtNRy-\x80 ") == b"acgtnnnnnn"


def test_refusals():
    with pytest.raises(FastaError, match="before the first header"):
        read_fasta(b"acgt\n>a\nacgt\n")
    with pytest.raises(FastaError, match="before the first header"):
        read_fasta(b"\n\n  ACGT")
    with pytest.raises(FastaError, match="gzip"):
        read_fasta(b"\x1f\x8b\x08\x00")
