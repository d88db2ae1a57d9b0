"""CPU-only: the host side of the best-hit search -- one SAM line per read (sam_lines_best_hit) and the BestHit rows."""
import numpy as np

from zoe_b200 import BestHit, MaybeAligned, Strand, _lib, reverse_complement
from zoe_b200.alignment import Alignment, CudaProfiles, _pack
from zoe_b200.sam import sam_lines_best_hit


def best_hit_arrays():
    """Hand-made align_best_hit_arrays output for four reads against two references: a forward winner with a
    runner-up, a reverse winner without one, an Unmapped read and an Overflowed read."""
    reads = [b"ACGTACGTAA", b"GGGTTTCCCA", b"NNNN", b"ACGTACGTACGT"]
    buf, offs = _pack(reads)
    a = {
        "hit": np.array([1, 0, 0, 1], np.uint32), "strand": np.array([0, 1, 0, 0], np.uint8),
        "score": np.array([18, 20, 0, 0], np.uint32),
        "status": np.array([_lib.SOME, _lib.SOME, _lib.UNMAPPED, _lib.OVERFLOWED], np.uint8),
        "tier": np.array([8, 8, 8, 8], np.uint8), "runner_up": np.array([7, 0, 0, 0], np.uint32),
        "ref_start": np.array([4, 10, 0, 0], np.uint32), "ref_end": np.array([13, 20, 0, 0], np.uint32),
        "query_start": np.array([0, 0, 0, 0], np.uint32), "query_end": np.array([10, 10, 0, 0], np.uint32),
        "hazard": np.zeros(4, np.uint8),
        "cigar": np.array([(9 << 4) | 0, (1 << 4) | 1, (10 << 4) | 0], np.uint32),
        "cigar_off": np.array([0, 2, 3, 3, 3], np.uint64),
    }
    return reads, buf, offs, a


def test_one_line_per_read():
    reads, buf, offs, a = best_hit_arrays()
    lines = list(sam_lines_best_hit(a, ["r0", "r1", "r2", "r3"], ["refA", "refB"], buf, offs,
                                    quals=[b"ABCDEFGHIJ", b"0123456789", b"!!!!", b"############"]))
    assert len(lines) == len(reads)
    f = [ln.split("\t") for ln in lines]
    assert [x[0] for x in f] == ["r0", "r1", "r2", "r3"]
    # forward winner: refB at ref_start + 1, its CIGAR, AS and XS
    assert f[0][1:6] == ["0", "refB", "5", "255", "9M1I"]
    assert f[0][9:] == ["ACGTACGTAA", "ABCDEFGHIJ", "AS:i:18", "XS:i:7"]
    # reverse winner: FLAG 16, reverse-complemented SEQ, reversed QUAL; no XS when the runner-up is 0
    assert f[1][1:6] == ["16", "refA", "11", "255", "10M"]
    assert f[1][9:] == [reverse_complement(reads[1]).decode(), "9876543210", "AS:i:20"]
    # not Some: unmapped records with RNAME *
    for x in f[2:]:
        assert x[1:6] == ["4", "*", "0", "255", "*"] and x[9:] == ["*", "*"]


def test_flag_and_without_quals():
    _, buf, offs, a = best_hit_arrays()
    f = [ln.split("\t") for ln in sam_lines_best_hit(a, ["a", "b", "c", "d"], ["x", "y"], buf, offs, flag=1, mapq=60)]
    assert f[0][1] == "1" and f[1][1] == "17" and f[0][4] == "60"
    assert f[0][10] == "*" and f[1][10] == "*"


def test_best_hit_rows():
    reads, _, _, a = best_hit_arrays()
    prof = CudaProfiles.__new__(CudaProfiles)  # the row builder needs only the targets and the orientation
    prof.targets = [b"A" * 30, b"C" * 25]
    prof.profiled_is_query = False
    rows = prof._best_hit_rows(reads, a)
    assert rows[0] == BestHit(1, Strand.Forward, MaybeAligned.some(Alignment(18, (4, 13), (0, 10), "9M1I", 25, 10)), 7)
    assert rows[1] == BestHit(0, Strand.Reverse, MaybeAligned.some(Alignment(20, (10, 20), (0, 10), "10M", 30, 10)), 0)
    assert rows[2] == BestHit(0, Strand.Forward, MaybeAligned.Unmapped, 0)
    assert rows[3] == BestHit(1, Strand.Forward, MaybeAligned.Overflowed, 0)
    prof.profiled_is_query = True
    assert prof._best_hit_rows(reads, a)[0].result.unwrap().ref_len == 10
