"""CPU-only: the host side of the paired-end best-hit search -- the FASTQ pair reader, the paired SAM records
(sam_lines_paired) and the synthetic read-pair generator."""
import numpy as np
import pytest

from zoe_b200 import _lib, reverse_complement, synth
from zoe_b200.alignment import _pack
from zoe_b200.fastq import pack_fastq_pairs, read_fastq_pairs
from zoe_b200.sam import sam_lines_paired


def fastq(*recs):
    return b"".join(b"@%s\n%s\n+\n%s\n" % (h, s, b"I" * len(s)) for h, s in recs)


# ---- FASTQ pairs ----
def test_fastq_pairs_match_names_and_strip_mate_suffix():
    r1 = fastq((b"p0/1 extra", b"ACGT"), (b"p1 1:N:0:1", b"GG"))
    r2 = fastq((b"p0/2", b"TTTT"), (b"p1 2:N:0:1", b"CCC"))
    assert [x[0] for x in read_fastq_pairs(r1, r2)] == ["p0", "p1"]
    names, buf1, offs1, q1, buf2, offs2, q2 = pack_fastq_pairs(r1, r2)
    assert names == ["p0", "p1"]
    assert bytes(buf1[:int(offs1[-1])]) == b"ACGTGG" and offs1.tolist() == [0, 4, 6]
    assert bytes(buf2[:int(offs2[-1])]) == b"TTTTCCC" and offs2.tolist() == [0, 4, 7]
    assert q1 == [b"IIII", b"II"] and q2 == [b"IIII", b"III"]


def test_fastq_pairs_count_mismatch():
    r1 = fastq((b"a", b"AC"), (b"b", b"AC"))
    r2 = fastq((b"a", b"AC"))
    with pytest.raises(ValueError, match="record count"):
        list(read_fastq_pairs(r1, r2))
    with pytest.raises(ValueError, match="record count"):
        pack_fastq_pairs(r2, r1)


def test_fastq_pairs_name_mismatch():
    with pytest.raises(ValueError, match="names differ"):
        list(read_fastq_pairs(fastq((b"a/1", b"AC")), fastq((b"b/2", b"AC"))))
    with pytest.raises(ValueError, match="names differ"):  # only a trailing /1 or /2 is a mate suffix
        list(read_fastq_pairs(fastq((b"a/3", b"AC")), fastq((b"a/2", b"AC"))))


# ---- SAM records ----
def paired_arrays():
    """Hand-made align_paired_best_hit_arrays output for four pairs against two references:
    0: proper, mate 1 forward at 11, mate 2 reverse at 101 (FLAG 99 / 147);
    1: proper, mate 1 reverse at 201, mate 2 forward at 51 (83 / 163);
    2: mate 1 forward at 31, mate 2 Unmapped (73 / 133);
    3: both Unmapped (77 / 141)."""
    m1 = [b"ACGTACGTAA", b"GGGTTTCCCA", b"ACGTAAAAAA", b"NNNN"]
    m2 = [b"TTGGCCAATT", b"CCCAAAGGGT", b"GATTACA", b""]
    buf1, offs1 = _pack(m1)
    buf2, offs2 = _pack(m2)
    S, U = _lib.SOME, _lib.UNMAPPED
    a = {
        "hit": np.array([1, 0, 1, 0], np.uint32), "proper": np.array([1, 1, 0, 0], np.uint8),
        "tlen": np.array([100, -160, 0, 0], np.int32),
        "strand": np.array([0, 1, 1, 0, 0, 1, 0, 1], np.uint8),
        "score": np.array([20, 18, 20, 19, 20, 0, 0, 0], np.uint32),
        "status": np.array([S, S, S, S, S, U, U, U], np.uint8),
        "runner_up": np.array([5, 0, 0, 0, 0, 0, 0, 0], np.uint32),
        "ref_start": np.array([10, 100, 200, 50, 30, 0, 0, 0], np.uint32),
        "ref_end": np.array([20, 110, 210, 60, 40, 0, 0, 0], np.uint32),
        "cigar": np.array([10 << 4] * 5, np.uint32),
        "cigar_off": np.array([0, 1, 2, 3, 4, 5, 5, 5, 5], np.uint64),
    }
    return m1, m2, buf1, offs1, buf2, offs2, a


def records():
    m1, m2, buf1, offs1, buf2, offs2, a = paired_arrays()
    q1 = [b"A" * len(s) for s in m1]
    q2 = [bytes(range(65, 65 + len(s))) for s in m2]
    lines = list(sam_lines_paired(a, ["p0", "p1", "p2", "p3"], ["refA", "refB"], buf1, offs1, buf2, offs2, q1, q2))
    return m1, m2, [ln.split("\t") for ln in lines]


def test_two_records_per_pair_mate1_first():
    _, _, f = records()
    assert len(f) == 8
    assert [x[0] for x in f] == ["p0", "p0", "p1", "p1", "p2", "p2", "p3", "p3"]
    assert [int(x[1]) & 0xC0 for x in f] == [0x40, 0x80] * 4


def test_proper_pair_flags_mates_and_tlen():
    m1, m2, f = records()
    # pair 0: 99 / 147, RNEXT = and PNEXT at the mate's POS, TLEN +100 / -100
    assert f[0][1:9] == ["99", "refB", "11", "255", "10M", "=", "101", "100"]
    assert f[1][1:9] == ["147", "refB", "101", "255", "10M", "=", "11", "-100"]
    assert f[0][9:] == [m1[0].decode(), "A" * 10, "AS:i:20", "XS:i:5"]
    assert f[1][9:] == [reverse_complement(m2[0]).decode(), "JIHGFEDCBA", "AS:i:18"]
    # pair 1: mate 1 reverse -> 83 / 163; mate 1's TLEN is negative (it starts after mate 2)
    assert f[2][1:9] == ["83", "refA", "201", "255", "10M", "=", "51", "-160"]
    assert f[3][1:9] == ["163", "refA", "51", "255", "10M", "=", "201", "160"]


def test_mapped_with_unmapped_mate():
    _, m2, f = records()
    # mate 1 mapped forward, mate 2 Unmapped: 73 / 133; the unmapped mate takes its mate's RNAME and POS and keeps
    # its SEQ and QUAL as given
    assert f[4][1:9] == ["73", "refB", "31", "255", "10M", "=", "31", "0"]
    assert f[5][1:9] == ["133", "refB", "31", "255", "*", "=", "31", "0"]
    assert f[5][9:] == [m2[2].decode(), "ABCDEFG"]


def test_unmapped_pair():
    m1, _, f = records()
    assert f[6][1:9] == ["77", "*", "0", "255", "*", "*", "0", "0"]
    assert f[7][1:9] == ["141", "*", "0", "255", "*", "*", "0", "0"]
    assert f[6][9] == m1[3].decode() and f[7][9:] == ["*", "*"]  # a 0-length mate has SEQ and QUAL *


def test_unmapped_mate1_reverse_mate2_flags():
    m1, m2, buf1, offs1, buf2, offs2, a = paired_arrays()
    a = {k: v.copy() for k, v in a.items()}
    a["status"][2], a["status"][3] = _lib.UNMAPPED, _lib.SOME  # pair 1: mate 1 unmapped, mate 2 mapped reverse
    a["strand"][3] = 1
    a["proper"][1], a["tlen"][1] = 0, 0
    f = [ln.split("\t") for ln in sam_lines_paired(a, list("abcd"), ["refA", "refB"], buf1, offs1, buf2, offs2)]
    assert f[2][1:9] == ["101", "refA", "51", "255", "*", "=", "51", "0"]  # 1 + 4 + 0x20 + 0x40
    assert f[3][1:9] == ["153", "refA", "51", "255", "10M", "=", "51", "0"]  # 1 + 8 + 0x10 + 0x80


# ---- synthetic pairs ----
def test_paired_reads_opposite_strands_and_insert():
    rng = np.random.default_rng(0)
    targets = [synth.random_dna(rng, L) for L in (900, 1200, 640)]
    m1, m2, t = synth.paired_reads(np.random.default_rng(1), targets, 400, read_len=100, insert_mean=300,
                                   insert_sd=40, sub=0.0, indel=0.0, random_frac=0.0)
    assert m1.shape == m2.shape == (400, 100)
    assert set(np.unique(t["strand"])) == {0, 1}
    for i in range(400):
        ref = bytes(targets[int(t["target"][i])])
        s, L = int(t["start"][i]), int(t["insert"][i])
        assert 100 <= L <= len(ref)
        a, b = bytes(m1[i]), bytes(m2[i])
        if t["strand"][i] == 0:  # mate 1 forward at the fragment start, mate 2 reverse at its end
            assert ref[s:s + 100] == a and ref[s + L - 100:s + L] == reverse_complement(b)
        else:  # the fragment is the other strand: mate 2 forward at the start, mate 1 reverse at the end
            assert ref[s:s + 100] == b and ref[s + L - 100:s + L] == reverse_complement(a)


def test_paired_reads_error_model_and_random_fraction():
    rng = np.random.default_rng(2)
    targets = [synth.random_dna(rng, 2000)]
    m1, m2, t = synth.paired_reads(np.random.default_rng(3), targets, 4000, read_len=150, insert_mean=400, insert_sd=60)
    ref = bytes(targets[0])
    exact = sum(bytes(m1[i]) == ref[int(t["start"][i]):int(t["start"][i]) + 150] for i in range(4000)
                if t["strand"][i] == 0)
    fwd = int((t["strand"] == 0).sum())
    # a read is exact with probability ~0.99^150 * 0.95 ~ 0.21
    assert 0.12 * fwd < exact < 0.32 * fwd
    assert abs(float(np.mean(t["insert"])) - 400) < 5
