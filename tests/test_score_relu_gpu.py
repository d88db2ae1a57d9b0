"""The score kernels' true-gap-state recurrence (sw_score.cuh): dW = diag + W, H = max(dW, E, F, 0), the gap states
opened from H - go, and the running maximum taken over dW.  Zero initial gap states, the per-half adds of the packed
kernels and the overflow detection through dW are exact only under the conditions DESIGN.md section 4 proves; these tests
hold them against the oracle where they are tightest:

  * gap penalties of zero (no gap costs anything, so a gap state equals the H it was opened from) and a tie-heavy
    scoring, in every row bucket of sw_score_kernel with one and with two column streams;
  * packed tasks whose one half overflows while the other scores small, and scores one below, at and one above the
    packed overflow threshold, in the single-pass, shared-rows and long-row kernels (the flagged halves are re-run by
    the 32-bit kernels);
  * the shared-rows and long-row kernels on the edge scorings;
  * the compiled headline kernel, read from the library: the adds stay per-half VIADD.16x2, not fused back into the
    max instructions."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from test_instantiation_sweep_gpu import (AA, ROW_BUCKETS, ROWS_KERNEL_K, ROWS_STREAM_MIN_LEN, SCORE_KERNELS, W25, W42,
                                          bucket_inputs, packed_overflow_threshold, port_score, protein_batch)
from zoe_b200 import BLOSUM_62, DNA_PROFILE_MAP, CudaProfiles, WeightMatrix, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.environ.get("ZOE_CUDA_LIB") or os.path.join(ROOT, "zoe_b200", "libzoe_cuda.so")

# (go, ge): both penalties zero, a free extension, and the tie-heavy penalties (with W42: match 4, mismatch -2)
EDGE_GAPS = [(0, 0), (-10, 0), (-3, -1)]
W127 = WeightMatrix.new(DNA_PROFILE_MAP, 127, -1, b"N")  # mismatches cost 1: scores land on every integer near 127 n
P127 = WeightMatrix(BLOSUM_62.mapping, np.where(np.eye(25, dtype=bool), 127, -1).astype(np.int8))
T127 = packed_overflow_threshold(127)  # 32639 = 127 * 257


def check(targets, reads, wm, go, ge, what):
    buf, offs = synth.pack(reads)
    prof = CudaProfiles.new_with_w256([bytes(t) for t in targets], wm, go, ge)
    got = prof.sw_score_arrays(buf, offs)
    st = prof.last_stats()
    prof.close()
    for g, w, name in zip(got, port_score(targets, buf, offs, wm, go, ge), ("score", "status", "tier")):
        assert np.array_equal(g, w), (what, name)
    return got, st


def straddle_reads(a, c):
    """Reads of symbol `a` (self-match 127) scoring T - 1, T and T + 1 against a long run of `a`; mismatches `c` cost 1.
    Each appears in the low and in the high half of a packed task (sequences 2t and 2t + 1 share one)."""
    below = [a] * 128 + [c] + [a] * 129   # 127 * 257 - 1
    at = [a] * 257                         # 127 * 257
    above = [a, c] * 126 + [a] * 132       # 127 * 258 - 126
    mk = lambda s: np.frombuffer(bytes(s), dtype=np.uint8).copy()  # noqa: E731
    return [mk(below), mk(at), mk(above), mk(below), mk(at), mk(above)]


def split_reads(rng, a, alphabet):
    """Packed tasks (big, small) and (small, big): one half overflows, the other must stay exact."""
    big = np.full(300, a, np.uint8)
    small = [alphabet[rng.integers(0, len(alphabet), n)] for n in (40, 90, 150)]
    return [big, small[0], small[1], big, big, small[2], big.copy()]


@pytest.mark.gpu
@pytest.mark.parametrize("G,K", SCORE_KERNELS)
def test_score_buckets_edge_gap_penalties(G, K):
    cap = G * K
    prev = max([b for b in ROW_BUCKETS if b < cap], default=0)
    targets, reads = bucket_inputs(cap, prev, 31, seed=cap + 77)
    for go, ge in EDGE_GAPS:
        wm = W42 if (go, ge) == (-3, -1) else W25
        for tset in (targets[:1], targets):  # one column stream, two
            check(tset, reads, wm, go, ge, (cap, go, ge, len(tset)))


@pytest.mark.gpu
@pytest.mark.parametrize("go,ge", [(-10, -1), (-11, -1), (0, 0)])  # compiled-in penalties, run-time ones, none
def test_score_packed_halves_and_threshold(go, ge):
    rng = np.random.default_rng(91)
    tgt = np.full(400, ord("A"), np.uint8)
    for tset in ([tgt], [tgt, synth.random_dna(rng, 90)]):
        got, st = check(tset, split_reads(rng, ord("A"), np.frombuffer(b"ACGT", np.uint8)), W127, go, ge, (go, "split"))
        assert int(got[0][0, 0]) == 127 * 300 and st["rerun_wide"] > 0
        reads = straddle_reads(ord("A"), ord("C")) + [synth.random_dna(rng, 120)]
        got, st = check(tset, reads, W127, go, ge, (go, "straddle"))
        if (go, ge) != (0, 0):  # a free gap skips the mismatch instead
            assert [int(s) for s in got[0][:6, 0]] == [T127 - 1, T127, T127 + 1] * 2
        assert st["rerun_wide"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("K", ROWS_KERNEL_K)
def test_rows_kernels_edge_cases(K):
    """sw_score_rows*_kernel<32, K>: shortest streamed 64 takes the streaming variant, 63 the other one."""
    rng = np.random.default_rng(700 + K)
    targets = [AA[rng.integers(0, 20, 32 * K)], AA[rng.integers(0, 20, 45)]]
    for shortest in (ROWS_STREAM_MIN_LEN, ROWS_STREAM_MIN_LEN - 1):
        lens = [shortest, 700, shortest + 1, 32 * K] + [int(x) for x in rng.integers(shortest, 701, 13)]
        reads = protein_batch(rng, targets, lens)
        for go, ge in EDGE_GAPS:
            check(targets, reads, BLOSUM_62, go, ge, (K, shortest, go, ge))
    # overflow: the profiled run of 'A' (it picks the kernel) has to hold the 384-residue straddling read; a random
    # protein keeps the alphabet large enough for the shared-rows path
    if 32 * K >= 384:
        tset = [np.full(32 * K, ord("A"), np.uint8), AA[rng.integers(0, 20, 200)]]
        for go, ge in ((-10, -1), (0, 0)):
            got, st = check(tset, split_reads(rng, ord("A"), AA), P127, go, ge, (K, go, "split"))
            assert int(got[0][0, 0]) == 127 * 300 and st["rerun_wide"] > 0
            reads = straddle_reads(ord("A"), ord("C")) + [AA[rng.integers(0, 20, 130)]]
            got, st = check(tset, reads, P127, go, ge, (K, go, "straddle"))
            if go:
                assert [int(s) for s in got[0][:6, 0]] == [T127 - 1, T127, T127 + 1] * 2


@pytest.mark.gpu
def test_long_kernel_edge_cases():
    """Streamed sequences over 1024 rows take sw_score_long_kernel: rows in chunks, (H, E) parked between them."""
    rng = np.random.default_rng(313)
    targets = [synth.random_dna(rng, 1800), synth.random_dna(rng, 300)]
    src = targets[0]
    reads = [src[100:1500].copy(), synth.random_dna(rng, 1100), src[:1025].copy(), src[700:1800][::-1].copy(),
             synth.random_dna(rng, 2200), src[50:1700].copy(), synth.random_dna(rng, 40)]
    reads[3][::7] = ord("G")
    for go, ge in EDGE_GAPS:
        check(targets, reads, W42 if (go, ge) == (-3, -1) else W25, go, ge, ("long", go, ge))
    # overflow in the long kernel: bound min(1100, 400) x 127 stays packed, so the flagged halves are re-run
    tgt = np.full(400, ord("A"), np.uint8)
    for go, ge in ((-10, -1), (0, 0)):
        tset = [tgt, synth.random_dna(rng, 90)]
        got, st = check(tset, split_reads(rng, ord("A"), np.frombuffer(b"ACGT", np.uint8)) + [synth.random_dna(rng, 1100)],
                        W127, go, ge, ("long split", go))
        assert int(got[0][0, 0]) == 127 * 300 and st["rerun_wide"] > 0
        reads = straddle_reads(ord("A"), ord("C")) + [synth.random_dna(rng, 1100)]
        got, st = check(tset, reads, W127, go, ge, ("long straddle", go))
        if go:
            assert [int(s) for s in got[0][:6, 0]] == [T127 - 1, T127, T127 + 1] * 2


HEADLINE = "_ZN8zoe_cuda15sw_score_kernelILi8ELi19ELb1ELi2ENS_6GapImmILi10ELi1EEELb1EEEvNS_11ScoreParamsE"


def headline_sass():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(LIB) or not os.path.exists(exe):
        pytest.skip("needs the built library and cuobjdump")
    lines, inside = [], False
    with subprocess.Popen([exe, "-sass", LIB], stdout=subprocess.PIPE, text=True) as proc:
        for line in proc.stdout:
            if "Function : " in line:
                if inside:
                    break
                inside = line.split("Function : ")[1].strip() == HEADLINE
            elif inside:
                lines.append(line)
        proc.kill()
    assert lines, HEADLINE + " not found in " + LIB
    return "".join(lines)


def test_headline_kernel_keeps_the_per_half_adds():
    """cfg 2's kernel: dW and H - go are VIADD.16x2 (off the ALU pipe); ptxas has not fused them back into
    VIADDMNMX.S16x2.RELU, which would put the row back at 4.5 ALU-pipe instructions per cell pair."""
    sass = headline_sass()
    ops = re.findall(r"\b(VIADD\.16x2|VIADDMNMX\.S16x2\.RELU|VIADDMNMX\.S16x2|VIMNMX3\.S16x2\.RELU)\b", sass)
    assert ops.count("VIADD.16x2") >= 2 * 19 * 2  # two per row, 19 rows, two streams: at least one column step
    assert ops.count("VIMNMX3.S16x2.RELU") >= 19 * 2
    assert "VIADDMNMX.S16x2.RELU" not in ops
