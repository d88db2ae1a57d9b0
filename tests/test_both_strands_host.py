"""CPU only: the host side of the both-strand search -- the Strand enum, the Python complement table and the SAM
records of reverse-strand results."""
import numpy as np

from zoe_b200 import Alignment, MaybeAligned, Strand, reverse_complement
from zoe_b200.sam import sam_lines_from_arrays, sam_records

# the complement table, written out from its specification
_PAIRS = {"A": "T", "T": "A", "U": "A", "C": "G", "G": "C", "R": "Y", "Y": "R", "K": "M", "M": "K", "B": "V", "V": "B",
          "D": "H", "H": "D", "S": "S", "W": "W", "N": "N"}


def expected_complement(b: int) -> int:
    c = chr(b)
    if c in _PAIRS:
        return ord(_PAIRS[c])
    if c.upper() in _PAIRS and c.islower():
        return ord(_PAIRS[c.upper()].lower())
    return b


def test_reverse_complement_maps_every_byte_by_the_table():
    for b in range(256):
        assert reverse_complement(bytes([b])) == bytes([expected_complement(b)]), b
    every = bytes(range(256))
    assert reverse_complement(every) == bytes(expected_complement(b) for b in reversed(every))


def test_reverse_complement_examples():
    assert reverse_complement(b"") == b""
    assert reverse_complement(b"ACGTN") == b"NACGT"
    assert reverse_complement(b"acgu") == b"acgt"
    assert reverse_complement(b"AAGCTT") == b"AAGCTT"  # a palindrome
    assert reverse_complement(bytearray(b"RYKMBVDH")) == b"DHBVKMRY"


def test_strand_enum():
    assert Strand.Forward.value == 0 and Strand.Reverse.value == 1
    assert Strand(1) is Strand.Reverse


def _result():
    a0 = Alignment(10, (2, 7), (0, 5), "5M", 20, 5)
    a1 = Alignment(8, (4, 8), (1, 5), "1S4M", 20, 5)
    return [[MaybeAligned.some(a0), MaybeAligned.Unmapped], [MaybeAligned.some(a1), MaybeAligned.some(a0)]]


def test_sam_records_reverse_strand():
    seqs, quals = [b"ACGTT", b"GGCAT"], [b"ABCDE", b"FGHIJ"]
    plain = [str(r) for r in sam_records(_result(), ["r0", "r1"], ["t0", "t1"], seqs, quals)]
    fwd = [[Strand.Forward] * 2] * 2
    assert [str(r) for r in sam_records(_result(), ["r0", "r1"], ["t0", "t1"], seqs, quals, strand=fwd)] == plain
    strand = [[Strand.Forward, Strand.Reverse], [Strand.Reverse, Strand.Forward]]
    recs = sam_records(_result(), ["r0", "r1"], ["t0", "t1"], seqs, quals, strand=strand)
    assert [r.flag for r in recs] == [0, 4, 16, 0]  # unmapped records stay as they are
    assert (recs[2].seq, recs[2].qual, recs[2].cigar, recs[2].pos) == (b"ATGCC", b"JIHGF", "1S4M", 5)
    assert (recs[3].seq, recs[3].qual) == (b"GGCAT", b"FGHIJ")
    no_qual = sam_records(_result(), ["r0", "r1"], ["t0", "t1"], seqs, strand=strand)
    assert (no_qual[2].seq, no_qual[2].qual) == (b"ATGCC", b"*")


def test_sam_lines_from_arrays_reverse_strand():
    buf = np.frombuffer(b"ACGTTGGCAT", dtype=np.uint8)
    offs = np.array([0, 5, 10], dtype=np.uint64)
    a = {"status": np.array([0, 2], dtype=np.uint8), "score": np.array([10, 0], dtype=np.uint32),
         "ref_start": np.array([2, 0], dtype=np.uint32), "cigar": np.array([5 << 4], dtype=np.uint32),
         "cigar_off": np.array([0, 1, 1], dtype=np.uint64)}
    args = (a, 1, ["r0", "r1"], ["t0"], buf, offs, [b"ABCDE", b"FGHIJ"])
    plain = list(sam_lines_from_arrays(*args))
    assert list(sam_lines_from_arrays(*args, strand=None)) == plain
    assert list(sam_lines_from_arrays(*args, strand=np.zeros(2, dtype=np.uint8))) == plain
    rev = list(sam_lines_from_arrays(*args, strand=np.array([1, 1], dtype=np.uint8)))
    assert rev[0].split("\t")[:6] == ["r0", "16", "t0", "3", "255", "5M"]
    assert rev[0].split("\t")[9:11] == ["AACGT", "EDCBA"]
    assert rev[1] == plain[1]  # unmapped
