"""The plain Python FASTA / FASTQ parser (tests/fastx_truth.py) that the device parser is checked against, pinned on
hand-written inputs with hand-written answers: every rule it states, empty records, a headerless start, no final line
feed, CRLF, and blank lines at the end of a FASTQ file."""
import numpy as np
import pytest

from fastx_truth import NO_HEADER, parse

N = NO_HEADER

CASES = [
    # id, data, alphabet, fmt, sequence (alphabet characters), starts, header offsets, names
    ("fasta", b">a\nACGT\n>b\nGG\n", "dna4", 1, "ACGTGG", [0, 4, 6], [0, 8], ["a", "b"]),
    ("wrapped", b">x desc\nAC\nGT\nA\n", "dna4", 1, "ACGTA", [0, 5], [0], ["x desc"]),
    ("comments", b">a\n;note ACGN\nAC\n;x\nG\n", "dna4", 1, "ACG", [0, 3], [0], ["a"]),
    ("headerless start", b"ACG\n>r\nTT\n", "dna4", 1, "ACGTT", [0, 3, 5], [N, 4], ["", "r"]),
    ("no header at all", b"AC\nGT", "dna4", 1, "ACGT", [0, 4], [N], [""]),
    ("comment only", b";c\n", "dna4", 0, "", [0, 0], [N], [""]),
    ("no final line feed", b">a\nAC\n>b\nGT", "dna4", 1, "ACGT", [0, 2, 4], [0, 6], ["a", "b"]),
    ("crlf", b">a\r\nAC\r\nG\r\n>b\r\nT\r\n", "dna4", 1, "ACGT", [0, 3, 4], [0, 11], ["a", "b"]),
    ("empty records", b">a\n>b\nAC\n>c\n>d\n", "dna4", 1, "AC", [0, 0, 2, 2, 2], [0, 3, 9, 12], ["a", "b", "c", "d"]),
    ("blank lines, tabs, spaces", b">a\n\nA C\tG\n\n T\r\n", "dna4", 1, "ACGT", [0, 4], [0], ["a"]),
    ("soft-masked", b">a\nacGt\n", "dna4", 1, "ACGT", [0, 4], [0], ["a"]),
    ("any byte in a header", b">\xff\x00N?\nAC\n", "dna4", 1, "AC", [0, 2], [0], ["\ufffd\x00N?"]),
    ("dna5", b">a\nACGNT\nn\n", "dna5", 0, "ACGNTN", [0, 6], [0], ["a"]),
    ("dna15", b">d\nABCDGHKMNRSTVWY\nry\n", "dna15", 1, "ABCDGHKMNRSTVWYRY", [0, 17], [0], ["d"]),
    ("aa27", b">p\nMK*\n>q\nwxyz\n", "aa27", 1, "MK*WXYZ", [0, 3, 7], [0, 7], ["p", "q"]),
    ("fastq", b"@a\nACGT\n+\nIIII\n@b\nGG\n+\nII\n", "dna4", 2, "ACGTGG", [0, 4, 6], [0, 15], ["a", "b"]),
    ("fastq by first byte", b"@a\nACGT\n+\nIIII\n", "dna4", 0, "ACGT", [0, 4], [0], ["a"]),
    ("fastq trailing blank line", b"@a\nACGT\n+\nIIII\n@b\nGG\n+\nII\n\n", "dna4", 2, "ACGTGG", [0, 4, 6], [0, 15], ["a", "b"]),
    ("fastq trailing blank lines", b"@a\nAC\n+\nII\n\n\n\n\n\n", "dna4", 2, "AC", [0, 2], [0], ["a"]),
    ("fastq crlf, trailing blank line", b"@a\r\nAC\r\n+\r\nII\r\n\r\n", "dna4", 2, "AC", [0, 2], [0], ["a"]),
    ("fastq quality starts with @ and +", b"@a\nAC\n+\n@+\n@b\nG\n+\n+\n", "dna4", 2, "ACG", [0, 2, 3], [0, 11], ["a", "b"]),
    ("fastq empty record", b"@a\n\n+\n\n@b\nAC\n+\nII\n", "dna4", 2, "AC", [0, 0, 2], [0, 7], ["a", "b"]),
    ("fastq no final line feed", b"@a\nAC\n+\nII\n@b\nG\n+\nI", "dna4", 0, "ACG", [0, 2, 3], [0, 11], ["a", "b"]),
]


@pytest.mark.parametrize("data,alphabet,fmt,seq,starts,headers,names", [c[1:] for c in CASES], ids=[c[0] for c in CASES])
def test_reference_parser(data, alphabet, fmt, seq, starts, headers, names):
    from kmer_index_b200 import ALPHABET_CHARS
    p = parse(data, alphabet, fmt)
    want = np.array([ALPHABET_CHARS[alphabet].index(c) for c in seq], dtype=np.uint8)
    assert np.array_equal(p.ranks, want)
    assert p.starts.tolist() == starts
    assert p.header_offsets.tolist() == headers
    assert p.names == names


REFUSED = [
    ("not in dna4", b">a\nACGN\n", "dna4", 1),
    ("'>' inside a sequence line", b">a\nAC>G\n", "dna4", 1),
    ("FASTQ read as FASTA", b"@a\nAC\n+\nII\n", "dna4", 1),
    ("fastq blank line between records", b"@a\nAC\n+\nII\n\n@b\nGG\n+\nII\n", "dna4", 2),
    ("fastq sequence not in dna5", b"@a\nACGX\n+\nIIII\n", "dna5", 0),
    ("unknown format", b">a\nAC\n", "dna4", 3),
    ("empty input", b"", "dna4", 0),
]


@pytest.mark.parametrize("data,alphabet,fmt", [c[1:] for c in REFUSED], ids=[c[0] for c in REFUSED])
def test_reference_parser_refuses(data, alphabet, fmt):
    with pytest.raises(ValueError):
        parse(data, alphabet, fmt)
